"""The projector tail (``ProjectorTailContrastive_ms``) on the device-driven path: the Philox sampler against the drop-in
class on the projected maps, native bf16 / fp16 and channels-last maps against the same module on their fp32 widening,
``torch.autocast``, the memory of a cfg-2 step with bf16 maps, CUDA-graph capture, and (without a device) the argument
checks of the raw row entry points.

Tolerances: sampling is compared exactly.  Between two runs of the tail on the same rows (half map against its exact fp32
widening, replay against eager), only the order of the similarity kernels' fp32 atomics differs: loss and terms within
2e-6 relative, dz within 3e-4 of its maximum plus one ulp of its type (test_gpu_graph._close_grad), dW and db within
1e-3 of their maximum (a sum over every sampled row).  Against the drop-in class on ``tail(z)`` the projection itself
differs (a library convolution on every pixel): loss within 1e-4 relative, gradient cosine >= 0.9999."""
import ctypes as C

import pytest
import torch

BASE = 2 ** 62
PH_CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
              cross_scale_contrast=True, min_views_per_class=5, max_views_per_class=40, max_features_total=600,
              sampler="philox", sampler_seed=7)
REF_CFG = {k: v for k, v in PH_CFG.items() if k not in ("sampler", "sampler_seed")}
C_PREV, D = 32, 64
_FAKE = 0x100000        # a 1 MiB-aligned address that is never dereferenced: validation fails first


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import mscs_b200
    assert mscs_b200.load().mscs_device_ok() == 1, "libmscs.so needs a compute-capability 10.x device"
    return torch.device("cuda:0")


def _inputs(r, dev, dtype=torch.float32, layout="nchw"):
    from mscs_b200 import synth
    labels = synth.synth_labels(2, 128, 256, 19, 6, 16, 0.05, 1)
    zs = synth.synth_features(2, C_PREV, 128, 256, [4, 8, 16], 10 + r)
    fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
    return labels.to(dev), [z.to(dev, dtype).contiguous(memory_format=fmt) for z in zs]


def _module(cfg, dev, seed=5):
    from mscs_b200 import ProjectorTailContrastive_ms
    torch.manual_seed(seed)
    return ProjectorTailContrastive_ms(dict(cfg), C_PREV, D).to(dev)


def _params(mod):
    return [t.weight for t in mod.tails] + [t.bias for t in mod.tails]


def _run(mod, labels, zs, grad=True):
    """Loss and the gradients w.r.t. the maps, weights and biases."""
    leaves = [z.detach().clone(memory_format=torch.preserve_format).requires_grad_(grad) for z in zs]
    with torch.set_grad_enabled(grad):
        loss = mod(labels, leaves)
        grads = torch.autograd.grad(loss, leaves + _params(mod)) if grad else None
    return loss.detach(), grads


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm()))


def _close_grad(g, ref, rel=3e-4):
    mant = {torch.float32: 23, torch.bfloat16: 7, torch.float16: 10}[ref.dtype]
    r = ref.float()
    tol = rel * r.abs().max().item() + r.abs() * 2.0 ** -mant
    assert bool(((g.float() - r).abs() <= tol).all()), float((g.float() - r).abs().max())


def _same_samples(a_mod, b_mod):
    for a, b in zip(a_mod.fetch_samples(), b_mod.fetch_samples()):
        assert (a.T, a.V, a.N) == (b.T, b.V, b.N)
        assert torch.equal(a.idx_ref, b.idx_ref) and torch.equal(a.pair_ref, b.pair_ref) and torch.equal(a.pix, b.pix)


def _same_loss(a_mod, b_mod, la, lb, rel=2e-6):
    assert abs(float(la) - float(lb)) <= rel * abs(float(lb)), (float(la), float(lb))
    ga, gb = a_mod.fetch_logged(), b_mod.fetch_logged()
    for k in ("ms_losses", "cs_losses"):
        assert len(ga[k]) == len(gb[k]) and ga[k]
        for x, y in zip(ga[k], gb[k]):
            assert abs(x - y) <= rel * abs(y), (k, x, y)
    assert ga["has_inf_or_nan"] is False


def _check_grads(grads, ref, zs, S=3):
    for s in range(S):
        g, r = grads[s], ref[s]
        assert g.dtype == zs[s].dtype and g.shape == zs[s].shape and g.stride() == zs[s].stride()
        _close_grad(g, r.to(g.dtype))
    for g, r in zip(grads[S:], ref[S:]):
        _close_grad(g, r, 1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_philox_matches_dropin_on_projected_maps(layout, dev):
    import mscs_b200
    mod = _module(PH_CFG, dev)
    labels, zs = _inputs(0, dev, layout=layout)
    rng = torch.get_rng_state()
    mod._sampler_calls = 3
    loss, grads = _run(mod, labels, zs)
    drop = mscs_b200.DenseContrastiveLossV2_ms(dict(PH_CFG))
    drop._sampler_calls = 3
    leaves = [z.detach().clone(memory_format=torch.preserve_format).requires_grad_(True) for z in zs]
    dloss = drop(labels, [t(z) for t, z in zip(mod.tails, leaves)])
    dgrads = torch.autograd.grad(dloss, leaves + _params(mod))
    torch.cuda.synchronize()
    assert torch.equal(rng, torch.get_rng_state())
    _same_samples(mod, drop)
    dloss = dloss.detach()
    assert abs(float(loss) - float(dloss)) <= 1e-4 * abs(float(dloss))
    for s in range(3):
        assert torch.equal((grads[s] != 0).any(dim=1), (dgrads[s] != 0).any(dim=1)), "different gradient pixels"
        assert grads[s].stride() == zs[s].stride()
    for g, r in zip(grads, dgrads):
        assert _cos(g, r) >= 0.9999


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_half_maps_read_natively(layout, dtype, dev):
    mod, ref = _module(PH_CFG, dev), _module(PH_CFG, dev)
    labels, zs = _inputs(0, dev, dtype, layout)
    mod._sampler_calls = ref._sampler_calls = 1
    loss, grads = _run(mod, labels, zs)
    rloss, rgrads = _run(ref, labels, [z.float() for z in zs])
    _same_samples(mod, ref)
    _same_loss(mod, ref, loss, rloss)
    _check_grads(grads, rgrads, zs)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_autocast(dtype, dev):
    """Under autocast the GEMMs of the tail still run in fp32 (reference sampler: the path users run)."""
    mod = _module(REF_CFG, dev)
    labels, zs = _inputs(0, dev, dtype)
    torch.manual_seed(11)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss, grads = _run(mod, labels, zs)
    ref = _module(REF_CFG, dev)
    torch.manual_seed(11)
    rloss, rgrads = _run(ref, labels, [z.float() for z in zs])
    _same_samples(mod, ref)
    _same_loss(mod, ref, loss, rloss)
    _check_grads(grads, rgrads, zs)


@pytest.mark.gpu
def test_memory_cfg2_bf16(dev):
    """cfg-2 shape, bf16 NCHW maps: forward + backward allocate the bf16 dz and the GEMM rows, no fp32 copy of a map."""
    from mscs_b200 import ProjectorTailContrastive_ms, synth
    cfg = dict(synth.CONFIGS["cfg2"]["loss"])
    labels = synth.synth_labels(12, 512, 1024, 19, 19, 32, 0.05, 0).to(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    zs = [torch.randn(12, 256, 512 // s, 1024 // s, device=dev, generator=g).to(torch.bfloat16) for s in (4, 8, 16, 32)]
    torch.manual_seed(2)
    mod = ProjectorTailContrastive_ms(cfg, 256, 256).to(dev)
    leaves = [z.requires_grad_(True) for z in zs]
    for _ in range(2):          # warm-up: the workspace, cuBLAS handles
        torch.autograd.grad(mod(labels, leaves), leaves + _params(mod))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    grads = torch.autograd.grad(mod(labels, leaves), leaves + _params(mod))
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    e = mod.last_state.entry
    dz = sum(z.numel() * 2 for z in zs)
    ws = e.slab.numel() + 4 * (e.zd.numel() + e.P.numel()) + 4 * e.iota.numel()
    dZ = 4 * sum(N * 256 for N in mod.last_state.sp.Ncap)           # the GEMM's rows dZ
    bound = dz + ws + dZ + (16 << 20)
    fp32_copy = sum(z.numel() * 4 for z in zs)
    print(f"cfg2 bf16: peak {peak / 2**20:.1f} MiB, bound {bound / 2**20:.1f} MiB (dz {dz / 2**20:.1f}, "
          f"workspace {ws / 2**20:.1f}); an fp32 copy of the maps is {fp32_copy / 2**20:.1f} MiB")
    assert bound < dz + fp32_copy
    assert peak <= bound
    assert all(gz.dtype == torch.bfloat16 for gz in grads[:4])


def _capture(mod, st_lab, st_z, grad=True, lr=0.1):
    """Eager warm-up on a side stream, then the capture of forward (+ backward + an SGD step on the tails unless lr is
    None)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.set_grad_enabled(grad):
        loss = mod(st_lab, st_z)
        if grad:
            torch.autograd.grad(loss, st_z + _params(mod))
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    grads = None
    with torch.cuda.graph(g), torch.set_grad_enabled(grad):
        loss = mod(st_lab, st_z)
        if grad:
            grads = torch.autograd.grad(loss, st_z + _params(mod))
        if grad and lr is not None:
            with torch.no_grad():
                for p, gp in zip(_params(mod), grads[len(st_z):]):
                    p.sub_(lr * gp)
    return g, loss, grads


def _replay(g, st_lab, st_z, labels, zs):
    with torch.no_grad():
        st_lab.copy_(labels)
        for a, b in zip(st_z, zs):
            a.copy_(b)
    g.replay()


def _eager_at(mod, call, labels, zs, grad=True):
    ref = _module(PH_CFG, zs[0].device)
    ref.load_state_dict(mod.state_dict())
    ref._sampler_calls = call
    loss, grads = _run(ref, labels, zs, grad)
    return ref, loss, grads


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_captured_training_step_matches_eager(layout, dtype, dev):
    mod = _module(PH_CFG, dev)
    labels, zs = _inputs(0, dev, dtype, layout)
    st_lab = labels.clone()
    st_z = [z.clone(memory_format=torch.preserve_format).requires_grad_(True) for z in zs]
    g, loss, grads = _capture(mod, st_lab, st_z)
    assert mod._sampler_calls == 1 and int(mod.graph_call_index) == BASE
    rng = torch.get_rng_state()
    prev = None
    for r in range(3):
        _, fresh = _inputs(r + 1, dev, dtype, layout)
        before = {k: v.clone() for k, v in mod.state_dict().items()}
        ref = _module(PH_CFG, dev)
        ref.load_state_dict(before)
        _replay(g, st_lab, st_z, labels, fresh)
        ref._sampler_calls = BASE + r
        rloss, rgrads = _run(ref, labels, fresh)
        _same_samples(mod, ref)
        _same_loss(mod, ref, loss, rloss)
        _check_grads(grads, rgrads, zs)
        for p, q, gq in zip(_params(mod), _params(ref), rgrads[3:]):      # the captured SGD step (lr 0.1)
            want = q.detach() - 0.1 * gq
            assert float((p.detach() - want).abs().max()) <= 1e-4 * float(gq.abs().max()) + 1e-6 * float(want.abs().max())
        pix = [s.pix.clone() for s in mod.fetch_samples()]
        if prev is not None:
            assert any(not torch.equal(a, b) for a, b in zip(pix, prev)), "consecutive replays sampled the same pixels"
        prev = pix
    assert int(mod.graph_call_index) == BASE + 3 and mod._sampler_calls == 1
    assert torch.equal(rng, torch.get_rng_state())


@pytest.mark.gpu
def test_forward_only_capture_no_grad(dev):
    mod = _module(PH_CFG, dev)
    labels, zs = _inputs(0, dev)
    st_lab, st_z = labels.clone(), [z.clone() for z in zs]
    with torch.no_grad():
        g, loss, _ = _capture(mod, st_lab, st_z, grad=False)
    _, fresh = _inputs(1, dev)
    _replay(g, st_lab, st_z, labels, fresh)
    ref, rloss, _ = _eager_at(mod, BASE, labels, fresh, grad=False)
    _same_samples(mod, ref)
    _same_loss(mod, ref, loss, rloss)


@pytest.mark.gpu
def test_replay_without_pairs_then_recovery(dev):
    mod = _module(PH_CFG, dev)
    labels, zs = _inputs(0, dev)
    st_lab = labels.clone()
    st_z = [z.clone().requires_grad_(True) for z in zs]
    g, loss, grads = _capture(mod, st_lab, st_z, lr=None)
    _replay(g, st_lab, st_z, torch.full_like(labels, 19), zs)     # only the dropped last class: no pair is kept
    torch.cuda.synchronize()
    assert torch.isnan(loss).item() and float(mod.nan_flag) == 1.0
    assert all(int((x != 0).sum()) == 0 for x in grads[:3])
    with pytest.raises(RuntimeError, match="no \\(image, class\\) pair"):
        mod.fetch_logged()
    _, fresh = _inputs(1, dev)
    _replay(g, st_lab, st_z, labels, fresh)
    ref, rloss, rgrads = _eager_at(mod, BASE + 1, labels, fresh)
    _same_samples(mod, ref)
    _same_loss(mod, ref, loss, rloss)
    _check_grads(grads, rgrads, zs)
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
    from mscs_b200 import synth
    labels, zs = _inputs(0, dev)
    ref = _module(REF_CFG, dev)
    ref(labels, zs)
    _refused(lambda: ref(labels, zs))                                  # reference sampler
    fresh = _module(PH_CFG, dev)
    _refused(lambda: fresh(labels, zs))                                # no eager call before the capture
    mod = _module(PH_CFG, dev)
    mod(labels, zs)
    lab_cpu = labels.cpu()
    _refused(lambda: mod(lab_cpu, zs))                                 # labels not on the GPU
    odd = _module(PH_CFG, dev)
    lab_odd = synth.synth_labels(2, 120, 200, 19, 6, 4, 0.05, 1).to(dev)
    z_odd = [torch.randn(2, C_PREV, 120 // s, 200 // s, device=dev) for s in (4, 8, 8)]
    with pytest.raises(NotImplementedError):
        odd(lab_odd, z_odd)                                            # eager: as before
    _refused(lambda: odd(lab_odd, z_odd))                              # NCHW planes not a multiple of 8 pixels


# ---- without a device: the argument checks of the raw row entry points ----------------------------------------------
def _lib():
    import mscs_b200
    from mscs_b200 import _lib as L
    return mscs_b200.load(), L


def _gather_item(L, **kw):
    g = (L.GatherItem * 1)()
    g[0].feat = g[0].slot = g[0].anc_f32 = _FAKE
    g[0].n, g[0].C, g[0].plane = 1, 64, 8
    for k, v in kw.items():
        setattr(g[0], k, v)
    return g


def _rows_item(L, **kw):
    r = (L.RowsItem * 1)()
    r[0].feat = r[0].pix = r[0].dF = r[0].dfeat = r[0].anc_f32 = _FAKE
    r[0].rows, r[0].C, r[0].ldF = 1, 64, 64
    for k, v in kw.items():
        setattr(r[0], k, v)
    return r


def _dense_item(L, **kw):
    sc = (L.ScatterItem * 1)()
    sc[0].dF = sc[0].slot = sc[0].dfeat = _FAKE
    sc[0].ldF, sc[0].n, sc[0].C, sc[0].plane = 64, 1, 64, 8
    for k, v in kw.items():
        setattr(sc[0], k, v)
    return sc


def _rejected(rc, lib, what):
    assert rc < 0 and what in lib.mscs_last_error(), (rc, lib.mscs_last_error())


@pytest.mark.parametrize("bad", [-1, 3])
def test_raw_entry_points_reject_bad_dtype(bad):
    lib, L = _lib()
    _rejected(lib.mscs_gather_raw_batch(_gather_item(L, dtype=bad), 1, None), lib, b"dtype")
    _rejected(lib.mscs_gather_raw_rows_batch(_rows_item(L, dtype=bad), 1, None), lib, b"dtype")
    _rejected(lib.mscs_scatter_rows_nhwc_batch(_rows_item(L, dtype=bad, anc_f32=None), 1, None), lib, b"dtype")
    _rejected(lib.mscs_scatter_dense_batch(_dense_item(L, dtype=bad), (C.c_int32 * 1)(1), 1, None), lib, b"dtype")


def test_raw_entry_points_reject_null_pointers():
    lib, L = _lib()
    for f in ("feat", "slot", "anc_f32"):
        _rejected(lib.mscs_gather_raw_batch(_gather_item(L, **{f: None}), 1, None), lib, b"null pointer")
    for f in ("feat", "pix", "anc_f32"):
        _rejected(lib.mscs_gather_raw_rows_batch(_rows_item(L, **{f: None}), 1, None), lib, b"null pointer")
    for f in ("dF", "slot", "dfeat"):
        _rejected(lib.mscs_scatter_dense_batch(_dense_item(L, **{f: None}), (C.c_int32 * 1)(1), 1, None), lib,
                  b"null pointer")
    _rejected(lib.mscs_scatter_rows_nhwc_batch(_rows_item(L, anc_f32=None, pix=None), 1, None), lib, b"null pointer")
    _rejected(lib.mscs_scatter_rows_nhwc_batch(_rows_item(L, anc_f32=None, dF=None), 1, None), lib, b"gradient")


def test_half_null_normalisation_pair_is_rejected():
    lib, L = _lib()
    for kw in (dict(anc_f32=_FAKE), dict(inv_norm=_FAKE)):          # exactly one of the two set
        _rejected(lib.mscs_scatter_dense_batch(_dense_item(L, **kw), (C.c_int32 * 1)(1), 1, None), lib, b"both")
        r = _rows_item(L, anc_f32=kw.get("anc_f32"), inv_norm=kw.get("inv_norm"))
        _rejected(lib.mscs_scatter_rows_nhwc_batch(r, 1, None), lib, b"both")


@pytest.mark.parametrize("dtype", [1, 2], ids=["bf16", "fp16"])
def test_misaligned_half_gradients_are_rejected(dtype):
    lib, L = _lib()
    _rejected(lib.mscs_scatter_dense_batch(_dense_item(L, dtype=dtype, dfeat=_FAKE + 2), (C.c_int32 * 1)(1), 1, None),
              lib, b"aligned")
    _rejected(lib.mscs_scatter_rows_nhwc_batch(_rows_item(L, dtype=dtype, dfeat=_FAKE + 1, anc_f32=None), 1, None), lib,
              b"aligned")
