"""The pooled cross-batch mode with every input the single-process path takes as it is: bf16 / fp16 maps (no fp32 copy,
gradients in the map's dtype), channels-last maps (rows, no slot maps) and the Philox sampler.  Ranks are emulated on
one GPU (ThreadComm: the kernels, row ranges, peer-store gathers, statistics push and pull scatters of the pooled mode;
only the transport is local).

What the half path makes deterministic is compared exactly: sampling, and every rank's unit rows, inverse norms and
bf16 operand rows (a half element widens exactly, the arithmetic after the load is the fp32 kernel's).  Losses and
gradients go through the similarity kernels, whose atomics accumulate in an order that changes from run to run: those
are compared with tolerances (half vs fp32: loss 2e-6 relative, gradients 3e-4 of their maximum plus one ulp of the
half type; pooled vs single process: loss 2e-5 relative, gradient cosine > 0.99999).

The tests at the end (not marked gpu) check the gates and the argument validation of the pooled entry points without a
device."""
import threading

import pytest
import torch

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
LAYOUTS = ["nchw", "channels_last"]
CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
           cross_scale_contrast=True, w_high_low=0.5, w_high_mid=0.25, min_views_per_class=5,
           max_views_per_class=50, max_features_total=1500)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import mscs_b200
    assert mscs_b200.load().mscs_device_ok() == 1, "libmscs.so needs a compute-capability 10.x device"
    return torch.device("cuda:0")


def _inputs(n=4):
    """Labels and fp32 NCHW maps (CPU) of the small pooled case: several 128-row tiles per scale."""
    from mscs_b200 import synth
    return synth.synth_labels(n, 128, 256, 19, 7, 16, 0.05, 21), synth.synth_features(n, 64, 128, 256, [4, 8, 16], 22)


def _layout(x, layout):
    return x.contiguous(memory_format=torch.channels_last) if layout == "channels_last" else x.contiguous()


def _maps(feats, dtype, layout, dev):
    return [_layout(f.to(dev).to(dtype), layout) for f in feats]


def _samples(mod):
    return [(s.pix.clone(), s.pair_ref.clone(), s.idx_ref.clone()) for s in mod.last_samples]


def _same_pooled_samples(a, b, r, nl):
    """Rank r's sampling results of two pooled runs: pixels and pair lists whole, the reference-order indices of its own
    pairs (the rows of other ranks' pairs are never written on this rank)."""
    for (pix1, pair1, idx1), (pix2, pair2, idx2) in zip(a, b):
        assert torch.equal(pix1, pix2) and torch.equal(pair1, pair2)
        own = (pair1[:, 0] >= r * nl) & (pair1[:, 0] < (r + 1) * nl)
        assert torch.equal(idx1[own], idx2[own])


def _pooled_rows(st):
    """Per scale: this rank's fp32 unit rows and inverse norms (its own rows only: pix >= 0; the others are never
    written here) and the whole bf16 operand matrix in its exchange slab (every rank's rows), cloned."""
    sp = st.sp
    b = st.xs.keep[sp.x_off[st.par]["b"]:].view(torch.bfloat16)
    out = []
    for s, smp in enumerate(st.samples):
        N, Cc, mine = smp.N, sp.C, smp.pix >= 0
        out.append((st.fslab[sp.foff[s][0]:sp.foff[s][0] + N * Cc].view(N, Cc)[mine].clone(),
                    st.fslab[sp.foff[s][1]:sp.foff[s][1] + N][mine].clone(),
                    b[sp.boff[s]:sp.boff[s] + N * sp.C_pad].view(N, sp.C_pad).clone()))
    return out


def _single_rows(st):
    """The same three per scale from the single-process workspace (all rows)."""
    sp, e = st.sp, st.entry
    so = sp.slab_off
    bsl = e.slab[so["bslab"]:so["bslab"] + 2 * sp.bslab_n].view(torch.bfloat16)
    fsl = e.slab[so["fslab"]:so["fslab"] + 4 * sp.fslab_n].view(torch.float32)
    out = []
    for s, smp in enumerate(st.samples):
        N, Cc = smp.N, sp.C
        out.append((fsl[sp.foff[s][0]:sp.foff[s][0] + N * Cc].view(N, Cc).clone(),
                    fsl[sp.foff[s][1]:sp.foff[s][1] + N].clone(),
                    bsl[sp.boff[s]:sp.boff[s] + N * sp.C_pad].view(N, sp.C_pad).clone()))
    return out


def _pooled(cfg, labels, maps, world, seed, dev, calls=1, rows=True, mem=None):
    """`world` ranks emulated on this GPU, rank r passing images [r n/world, (r+1) n/world) of `labels` / `maps` (device
    tensors, any dtype and layout), `calls` forward + backward steps each.  The backward runs through
    _ops.run_backward, not loss.backward(): autograd runs every backward of one device on one engine thread, where the
    host barrier between emulated ranks would deadlock.  Returns per rank a list of per-call records.  `mem` (a dict):
    receives the device memory the last step allocated at peak over the memory allocated before it ("grew")."""
    import mscs_b200
    from mscs_b200 import _ops
    nl = labels.shape[0] // world
    shared = _ops.ThreadComm._Shared(world)
    results, errors = [None] * world, []

    def sync_all(fn):
        torch.cuda.synchronize()
        shared.barrier.wait()
        if fn is not None:
            fn()
        shared.barrier.wait()

    def worker(r):
        try:
            torch.cuda.set_device(dev)
            mod = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg), comm=_ops.ThreadComm(shared, r))
            lab = labels[r * nl:(r + 1) * nl]
            fts = [m[r * nl:(r + 1) * nl].detach().requires_grad_(True) for m in maps]
            recs = []
            for k in range(calls):
                measure = mem is not None and k == calls - 1
                if measure:
                    def start():
                        torch.cuda.reset_peak_memory_stats(dev)
                        mem["base"] = torch.cuda.memory_allocated(dev)
                    sync_all(start if r == 0 else None)
                loss = mod(lab, fts)
                st = mod.last_state
                grads = _ops.run_backward(st, torch.ones((), device=dev), [True] * len(fts),
                                          [tuple(f.shape) for f in fts], [f.dtype for f in fts])
                if measure:
                    sync_all((lambda: mem.update(grew=torch.cuda.max_memory_allocated(dev) - mem["base"]))
                             if r == 0 else None)
                torch.cuda.synchronize()
                recs.append(dict(loss=float(loss.detach()), grads=grads, samples=_samples(mod),
                                 terms=[float(x) for x in mod.ms_losses] + [float(x) for x in mod.cs_losses],
                                 rows=_pooled_rows(st) if rows else None))
                del loss, st
            results[r] = recs
        except Exception as e:      # noqa: BLE001
            errors.append(e)
            shared.barrier.abort()

    torch.manual_seed(seed)
    threads = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return results


def _single(cfg, labels, maps, seed, calls=1):
    """The single-process module on the whole batch, `calls` steps; per-call records as _pooled's."""
    import mscs_b200
    mod = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg))
    leaves = [m.detach().requires_grad_(True) for m in maps]
    torch.manual_seed(seed)
    recs = []
    for _ in range(calls):
        loss = mod(labels, leaves)
        grads = torch.autograd.grad(loss, leaves)
        recs.append(dict(loss=float(loss.detach()), grads=grads, samples=_samples(mod), rows=_single_rows(mod.last_state),
                         terms=[float(x) for x in mod.ms_losses] + [float(x) for x in mod.cs_losses]))
    return recs


def _close_grad(g, ref32, dtype):
    """g (half) against the fp32 path's gradient: 3e-4 of its maximum (run-to-run variation of the atomics) plus one
    ulp of the half type per element."""
    ref = ref32.to(dtype).float()
    mant = 7 if dtype == torch.bfloat16 else 10
    tol = 3e-4 * ref32.abs().max().item() + ref.abs() * 2.0 ** -mant + (2.0 ** -24 if dtype == torch.float16 else 0.0)
    assert bool(((g.float() - ref).abs() <= tol).all()), float((g.float() - ref).abs().max())


def _nonzero_pixels(g):
    return (g != 0).any(dim=1)


def _cosine(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / torch.sqrt((a @ a) * (b @ b)))


def _same_samples_as_single(rank_recs, single_rec, nl, planes):
    """Every sorted row is sampled by exactly one rank, at the single-process pixel of that row; pair lists are the
    same; the reference-order indices of a rank's own pairs are the single process's."""
    for s, plane in enumerate(planes):
        pix1, pair1, idx1 = single_rec["samples"][s]
        owner = torch.zeros_like(pix1)
        for r, rec in enumerate(rank_recs):
            pix, pair, idx = rec["samples"][s]
            assert torch.equal(pair, pair1)
            mine = pix >= 0
            owner += mine.int()
            assert torch.equal(pix[mine] + r * nl * plane, pix1[mine])
            own_pairs = (pair[:, 0] >= r * nl) & (pair[:, 0] < (r + 1) * nl)
            assert torch.equal(idx[own_pairs], idx1[own_pairs])
        assert bool((owner == 1).all())


def _matches_single(rank_recs, single_rec, nl, tol_loss=2e-5, min_cos=0.99999):
    want = single_rec["loss"]
    for r, rec in enumerate(rank_recs):
        assert abs(rec["loss"] - want) < tol_loss * abs(want), (r, rec["loss"], want)
        for a, b in zip(rec["terms"], single_rec["terms"]):
            assert abs(a - b) < tol_loss * abs(b)
        for s, g in enumerate(rec["grads"]):
            w = single_rec["grads"][s][r * nl:(r + 1) * nl]
            assert torch.equal(_nonzero_pixels(g), _nonzero_pixels(w)), f"rank {r} scale {s}: sampled pixels differ"
            cs = _cosine(g, w)
            print(f"rank {r} scale {s}: grad cosine {cs:.8f}")
            assert cs > min_cos


# ---- 1. pooled half maps against pooled fp32 on their exact widening ----------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("world", [2, 4])
def test_pooled_half_maps_match_pooled_fp32(world, dtype, layout, dev):
    labels, feats = _inputs()
    labels = labels.to(dev)
    maps = _maps(feats, DTYPES[dtype], layout, dev)
    nat = _pooled(CFG, labels, maps, world, 5, dev)
    rng_nat = torch.get_rng_state()
    ref = _pooled(CFG, labels, [m.float() for m in maps], world, 5, dev)
    assert torch.equal(rng_nat, torch.get_rng_state())
    nl = labels.shape[0] // world
    for r in range(world):
        a, b = nat[r][0], ref[r][0]
        _same_pooled_samples(a["samples"], b["samples"], r, nl)
        for x, y in zip(a["rows"], b["rows"]):        # unit rows, inverse norms, bf16 operand rows: bit for bit
            for u, v in zip(x, y):
                assert torch.equal(u, v)
        assert abs(a["loss"] - b["loss"]) <= 2e-6 * abs(b["loss"])
        for u, v in zip(a["terms"], b["terms"]):
            assert abs(u - v) <= 2e-6 * abs(v)
        for m, g, g32 in zip(maps, a["grads"], b["grads"]):
            mine = m[r * nl:(r + 1) * nl]
            assert g.dtype == m.dtype and g.shape == mine.shape and g.stride() == mine.stride()
            assert torch.equal(_nonzero_pixels(g), _nonzero_pixels(g32))
            _close_grad(g, g32, g.dtype)


# ---- 2. pooled against the single process on the concatenated batch ----------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_pooled_matches_single_process_every_dtype_and_layout(dtype, layout, dev):
    world = 2
    labels, feats = _inputs()
    labels = labels.to(dev)
    maps = _maps(feats, DTYPES[dtype], layout, dev)
    single = _single(CFG, labels, maps, 5)[0]
    assert single["samples"][0][0].numel() > 256          # several row tiles, so the row ranges matter
    res = _pooled(CFG, labels, maps, world, 5, dev, rows=False)
    nl = labels.shape[0] // world
    recs = [res[r][0] for r in range(world)]
    _same_samples_as_single(recs, single, nl, [f.shape[2] * f.shape[3] for f in feats])
    _matches_single(recs, single, nl)
    for r, rec in enumerate(recs):
        for m, g in zip(maps, rec["grads"]):
            assert g.dtype == m.dtype and g.stride() == m[r * nl:(r + 1) * nl].stride()


# ---- 3. channels-last pooled against NCHW pooled (fp32) -----------------------------------------------------------
@pytest.mark.gpu
def test_pooled_channels_last_matches_pooled_nchw(dev):
    """The channels-last gather keeps the lane / channel assignment of the single-process row gather, so its unit rows,
    inverse norms and bf16 operand rows are bit-identical to the single-process channels-last ones.  The NCHW pooled
    gather (k_gather_p2p) sums a lane's eight consecutive channels instead, so against it the unit rows and inverse
    norms agree to rounding (2e-6 relative), the sampled pixels exactly, and the loss within 2e-6 relative."""
    world = 2
    labels, feats = _inputs()
    labels = labels.to(dev)
    cl, nchw = _maps(feats, torch.float32, "channels_last", dev), _maps(feats, torch.float32, "nchw", dev)
    a = _pooled(CFG, labels, cl, world, 7, dev)
    b = _pooled(CFG, labels, nchw, world, 7, dev)
    single = _single(CFG, labels, cl, 7)[0]
    nl = labels.shape[0] // world
    for r in range(world):
        x, y = a[r][0], b[r][0]
        _same_pooled_samples(x["samples"], y["samples"], r, nl)
        for s, ((f1, i1, b1), (f2, i2, b2)) in enumerate(zip(x["rows"], y["rows"])):
            assert torch.allclose(f1, f2, rtol=2e-6, atol=1e-9) and torch.allclose(i1, i2, rtol=2e-6, atol=0)
            mine = x["samples"][s][0] >= 0
            f0, i0, b0 = single["rows"][s]
            assert torch.equal(f1, f0[mine]) and torch.equal(i1, i0[mine]) and torch.equal(b1, b0)
        assert abs(x["loss"] - y["loss"]) <= 2e-6 * abs(y["loss"])
        for g, h in zip(x["grads"], y["grads"]):
            assert g.is_contiguous(memory_format=torch.channels_last) and h.is_contiguous()
            assert torch.equal(_nonzero_pixels(g), _nonzero_pixels(h))
            assert _cosine(g, h) > 0.99999


# ---- 4. Philox: pooled against single process, two calls ----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("world,dtype,layout", [(2, "fp32", "nchw"), (4, "fp32", "nchw"), (2, "bf16", "channels_last")])
def test_pooled_philox_matches_single_process(world, dtype, layout, dev):
    cfg = dict(CFG, sampler="philox", sampler_seed=1234)
    labels, feats = _inputs()
    labels = labels.to(dev)
    maps = _maps(feats, DTYPES[dtype], layout, dev)
    single = _single(cfg, labels, maps, 3, calls=2)
    torch.manual_seed(3)
    before = torch.get_rng_state()
    res = _pooled(cfg, labels, maps, world, 3, dev, calls=2, rows=False)
    assert torch.equal(torch.get_rng_state(), before), "the pooled Philox sampler touched the torch CPU generator"
    nl = labels.shape[0] // world
    planes = [f.shape[2] * f.shape[3] for f in feats]
    for k in range(2):      # call index 0, then 1 on every rank
        recs = [res[r][k] for r in range(world)]
        _same_samples_as_single(recs, single[k], nl, planes)
        _matches_single(recs, single[k], nl)
    assert not torch.equal(single[0]["samples"][0][0], single[1]["samples"][0][0])    # the second call drew anew


# ---- 5. cfg-5 size, bf16 maps ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 8])
def test_pooled_cfg5_bf16(world, dev):
    """BASELINE config 5 (64 images, C = 256, planes 128x256 / 64x128 / 32x64 / 16x32) with bf16 maps.

    Memory bound.  The bf16 maps of all ranks hold M = 64 * 256 * 43520 * 2 B = 1426.1 MB.  The parent's route copied
    them to fp32 (2 M) and pre-zeroed fp32 dense gradients (2 M) in the forward, both alive at once, so its step
    allocated more than 4 M = 5704.3 MB over what was there before it.  The native route allocates the bf16 gradients
    (M) and each rank's per-call workspace, which the step plan sizes at about 265 MB here (fp32 unit rows 235.8 MB;
    index, slot and statistics buffers and the similarity workspace the rest): about 1.96 GB at world 2 and 3.55 GB at
    world 8 for all emulated ranks together.  The assertion is the parent's lower bound, 4 M."""
    import mscs_b200
    from mscs_b200 import synth
    cfg = dict(synth.CONFIGS["cfg5"]["loss"])
    labels, feats = synth.make_inputs("cfg5")
    labels = labels.to(dev)
    maps = [f.to(dev).to(torch.bfloat16) for f in feats]
    del feats
    M = sum(m.numel() * m.element_size() for m in maps)
    assert M == 64 * 256 * 43520 * 2
    single = _single(cfg, labels, maps, 0)[0]
    mem = {}
    res = _pooled(cfg, labels, maps, world, 0, dev, calls=2, rows=False, mem=mem)
    print(f"pooled cfg5 bf16 x{world}: step allocated {mem['grew'] / 1e6:.1f} MB at peak (bound {4 * M / 1e6:.1f} MB)")
    assert mem["grew"] < 4 * M
    nl = labels.shape[0] // world
    # the second call draws from the generator state the first left: compare the first call with the single process
    recs = [res[r][0] for r in range(world)]
    _same_samples_as_single(recs, single, nl, [m.shape[2] * m.shape[3] for m in maps])
    _matches_single(recs, single, nl, min_cos=0.99998)


@pytest.mark.gpu
def test_pooled_nchw_plane_not_multiple_of_8_still_refused(dev):
    """The host-driven order for NCHW planes that are not a multiple of 8 pixels stays single-process only."""
    import mscs_b200
    from mscs_b200 import _ops, synth
    labels = synth.synth_labels(2, 60, 100, 19, 6, 4, 0.05, 3).to(dev)
    f = synth.synth_features(2, 32, 60, 100, [4], 4)[0].to(dev).to(torch.bfloat16)     # 15 x 25 plane
    cfg = dict(CFG, scales=1, weights=[1.0], cross_scale_contrast=False)
    mod = mscs_b200.DenseContrastiveLossV2_ms(cfg, comm=_ops.ThreadComm(_ops.ThreadComm._Shared(2), 0))
    with pytest.raises(NotImplementedError, match="multiple of 8"):
        mod(labels[:1], [f[:1]])


# ---- no device: gates, argument validation, version ---------------------------------------------------------------
_FAKE = 0x100000        # a 1 MiB-aligned address that is never dereferenced: validation fails first


def _plan(world, shapes, nhwc):
    from mscs_b200 import _ops
    spec = _ops.LossSpec(num_classes=20, temperature=0.1, cs_temperature=0.1, weights=[1.0] * len(shapes))
    n, _, h, w = shapes[0]
    return spec, _ops._StepPlan(torch.device("cpu"), (n, 4 * h, 4 * w), shapes, spec, False, world, 0, nhwc)


def test_gates_accept_pooled_half_and_channels_last():
    from mscs_b200 import _ops
    shapes = [(2, 32, 16, 32), (2, 32, 8, 16)]
    spec, sp = _plan(2, shapes, False)
    assert _ops.half_io_ok(sp, 2)
    assert _ops.half_io_ok(_plan(2, shapes, True)[1], 2)
    assert not _ops.half_io_ok(_plan(2, [(2, 32, 15, 25)], False)[1], 2)      # host-driven planes: fp32 copy
    assert not _ops.fast_path_ok(spec, 2)                                     # still sequenced from Python
    cl = [torch.zeros(s).contiguous(memory_format=torch.channels_last) for s in shapes]
    assert _ops.channels_last_ok(spec, 2, cl) and _ops.channels_last_ok(spec, 8, cl)
    assert not _ops.channels_last_ok(spec, 2, [torch.zeros(s) for s in shapes])


def _peers():
    from mscs_b200 import _lib
    return _lib.ptr_array([_FAKE, 2 * _FAKE])


def _calls(feat=_FAKE, dfeat=_FAKE, pix=_FAKE, dtype=0):
    """Each pooled entry point with world 2, rank 0 and otherwise valid arguments."""
    import mscs_b200
    lib = mscs_b200.load()
    return {
        "gather_p2p": lambda: lib.mscs_gather_normalize_p2p(feat, 2, 64, 64, pix, 10, None, _peers(), 2, 0, 256, _FAKE,
                                                            _FAKE, None, dtype),
        "gather_rows_p2p": lambda: lib.mscs_gather_rows_p2p(feat, 64, pix, 10, None, _peers(), 2, 0, 256, _FAKE, _FAKE,
                                                            None, dtype),
        "scatter_sectors_pull": lambda: lib.mscs_scatter_sectors_pull(_peers(), 2, 256, 128, 64, _FAKE, _FAKE, pix, 2,
                                                                      64, 64, dfeat, None, dtype),
        "scatter_rows_pull": lambda: lib.mscs_scatter_rows_pull(_peers(), 2, 256, 128, 64, _FAKE, _FAKE, pix, 10, 64,
                                                                dfeat, None, dtype),
    }


@pytest.mark.parametrize("bad", [-1, 3])
@pytest.mark.parametrize("entry", ["gather_p2p", "gather_rows_p2p", "scatter_sectors_pull", "scatter_rows_pull"])
def test_pooled_entry_points_reject_bad_dtype(entry, bad):
    import mscs_b200
    lib = mscs_b200.load()
    assert _calls(dtype=bad)[entry]() < 0 and b"dtype" in lib.mscs_last_error()


@pytest.mark.parametrize("entry,dtype,offset", [("gather_p2p", 1, 1), ("gather_p2p", 0, 2), ("gather_rows_p2p", 2, 1),
                                                ("gather_rows_p2p", 0, 2), ("scatter_sectors_pull", 1, 8),
                                                ("scatter_sectors_pull", 0, 4), ("scatter_rows_pull", 2, 1),
                                                ("scatter_rows_pull", 0, 2)])
def test_pooled_entry_points_reject_misaligned_maps(entry, dtype, offset):
    """feat / dfeat aligned to the element size; the NCHW pull scatter's 16-byte stores need 16 bytes."""
    import mscs_b200
    lib = mscs_b200.load()
    assert _calls(feat=_FAKE + offset, dfeat=_FAKE + offset, dtype=dtype)[entry]() < 0
    assert b"aligned" in lib.mscs_last_error()


@pytest.mark.parametrize("entry", ["gather_p2p", "gather_rows_p2p", "scatter_sectors_pull", "scatter_rows_pull"])
@pytest.mark.parametrize("which", ["map", "index"])
def test_pooled_entry_points_reject_null_pointers(entry, which):
    import mscs_b200
    lib = mscs_b200.load()
    kw = dict(feat=None, dfeat=None) if which == "map" else dict(pix=None)
    assert _calls(**kw)[entry]() < 0 and b"null" in lib.mscs_last_error()


def test_pooled_entry_points_keep_rank_checks():
    import mscs_b200
    lib = mscs_b200.load()
    assert lib.mscs_gather_rows_p2p(_FAKE, 64, _FAKE, 10, None, _peers(), 2, 2, 256, _FAKE, _FAKE, None, 0) < 0
    assert b"rank" in lib.mscs_last_error()
    assert lib.mscs_gather_rows_p2p(_FAKE, 64, _FAKE, 10, None, _peers(), 2, 0, 8, _FAKE, _FAKE, None, 0) < 0
    assert b"offset" in lib.mscs_last_error()
    assert lib.mscs_scatter_rows_pull(_peers(), 9, 256, 128, 64, _FAKE, _FAKE, _FAKE, 10, 64, _FAKE, None, 0) < 0
    assert b"world" in lib.mscs_last_error()


def test_version_is_0_7_0():
    import mscs_b200
    assert mscs_b200.load().mscs_version().startswith(b"mscs 0.7.0 ")
