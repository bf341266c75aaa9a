"""The projector tail in the pooled cross-batch mode (``ProjectorTailContrastive_ms(config, c_prev, d, comm=...)``): the
compaction kernel ``mscs_local_rows_batch`` through the C ABI, and the pooled tail against the single-process tail on
the concatenated batch.  Ranks are emulated on one GPU (ThreadComm: the kernels, row ranges, peer stores, barriers and
pulls of the pooled mode; only the transport is local).

The compaction is compared exactly against a torch computation, with every output between guard regions.

Pooled against single process: sampling is compared exactly (pixels, pair lists, and the reference-order indices of a
rank's own pairs).  The operand rows are not bit-identical: each rank projects its own rows with a GEMM over M = its
local row count, the single process with M = the global row bound, and the library GEMM may split and order the
c_prev-long dot products differently for a different M.  The normalised rows then differ in the last bits, and the
similarity kernels' fp32 atomics add their own run-to-run order.  So the loss and terms are compared within 2e-5
relative, the gradient of each rank's z by cosine > 0.99999 (the pooled-vs-single tolerances of
test_gpu_pooled_io.py), and the sum over the ranks of dW and db within 1e-3 of their maximum (the tail's tolerance,
test_gpu_projector_tail.py).

The backward runs through projector._backward_pooled, not loss.backward(): autograd runs every backward of one device
on one engine thread, where the host barrier between emulated ranks would deadlock."""
import ctypes as C
import threading

import pytest
import torch

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
           cross_scale_contrast=True, w_high_low=0.5, w_high_mid=0.25, min_views_per_class=5,
           max_views_per_class=50, max_features_total=1500)
C_PREV, D = 32, 64
_FAKE = 0x100000        # a 1 MiB-aligned address that is never dereferenced: validation fails first
_GUARD = 0x5A5A5A5A


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import mscs_b200
    assert mscs_b200.load().mscs_device_ok() == 1, "libmscs.so needs a compute-capability 10.x device"
    return torch.device("cuda:0")


# ---- 1. the compaction kernel through the C ABI --------------------------------------------------------------------
def _guarded(n, dev, fill=_GUARD, g=1024):
    """An int32 buffer of n entries between two g-entry guard regions: (whole tensor, view of the n entries)."""
    t = torch.full((n + 2 * g,), fill, dtype=torch.int32, device=dev)
    t[g:g + n] = _GUARD
    return t, t[g:g + n]


def _case(kind, rows, plane, gen):
    """(pix, device count): the selection's pix array of one scale (rows entries) and its row count."""
    N = rows
    perm = torch.randperm(plane, generator=gen)[:rows].int()
    if kind == "all":
        pix = perm
    elif kind == "none":
        pix = torch.full((rows,), -1, dtype=torch.int32)
    elif kind == "blocks":          # alternating blocks of 128 rows, as the 128-row shards of the pooled mode
        pix = torch.where((torch.arange(rows) // 128) % 2 == 0, perm, torch.full_like(perm, -1))
    elif kind == "single":
        pix = torch.full((rows,), -1, dtype=torch.int32)
        pix[rows // 3] = perm[0]
    elif kind == "zero":            # N = 0: every entry is stale
        pix, N = perm, 0
    elif kind == "stale":           # a local row every third row below N; pixels above N must not be read
        N = rows // 2 + 5
        pix = torch.where(torch.arange(rows) % 3 == 0, perm, torch.full_like(perm, -1))
        pix[N:] = perm[N:]
    else:
        raise ValueError(kind)
    return pix, N


def _expect(pix, N, rows, slot):
    p = pix[:N].long()
    loc = p >= 0
    k = torch.cumsum(loc.long(), 0) - 1
    crow = torch.full((rows,), -1, dtype=torch.int32)
    crow[:N][loc] = k[loc].int()
    cpix = p[loc].int()
    slot2 = None
    if slot is not None:
        slot2 = slot.clone()
        slot2[cpix.long()] = torch.arange(cpix.numel(), dtype=torch.int32)
    return crow, cpix, slot2


def _run_local_rows(cases, dev, with_slot):
    """One mscs_local_rows_batch call over the scales `cases` = [(pix, N, plane)]; every output is checked exactly and
    every guard region (and every entry the call must not write) is checked unchanged."""
    import mscs_b200
    from mscs_b200 import _lib
    lib = mscs_b200.load()
    S = len(cases)
    keep, pix_d, n_d, crow, cpix, slots, slot_init = [], [], [], [], [], [], []
    for s, (pix, N, plane) in enumerate(cases):
        rows = pix.numel()
        pd = pix.to(dev)
        nd = torch.tensor([N], dtype=torch.int32, device=dev)
        cw, cv = _guarded(rows, dev)
        pw, pv = _guarded(rows, dev)         # cpix: room for every row; only n_local entries may be written
        keep += [pd, nd, cw, pw]
        pix_d.append(pd)
        n_d.append(nd)
        crow.append((cw, cv))
        cpix.append((pw, pv))
        if with_slot and s % 2 == 0:        # the selection's slot map: its row at every local pixel, -1 elsewhere
            init = torch.full((plane,), -1, dtype=torch.int32)
            loc = (torch.arange(rows) < N) & (pix >= 0)
            init[pix[loc].long()] = torch.arange(rows, dtype=torch.int32)[loc]
            sw, sv = _guarded(plane, dev)
            sv.copy_(init.to(dev))
            keep.append(sw)
            slots.append((sw, sv))
            slot_init.append(init)
        else:
            slots.append(None)
            slot_init.append(None)
    nw, nv = _guarded(S, dev)
    before = {id(t): t.clone() for t in keep + [nw]}
    rc = lib.mscs_local_rows_batch(_lib.ptr_array([t.data_ptr() for t in pix_d]),
                                   _lib.ptr_array([t.data_ptr() for t in n_d]),
                                   (C.c_int32 * S)(*[p.numel() for p, _, _ in cases]),
                                   _lib.ptr_array([v.data_ptr() for _, v in crow]),
                                   _lib.ptr_array([v.data_ptr() for _, v in cpix]),
                                   _lib.ptr_array([x[1].data_ptr() if x is not None else None for x in slots])
                                   if with_slot else None,
                                   nv.data_ptr(), S, None)
    assert rc == 0, lib.mscs_last_error()
    torch.cuda.synchronize()
    g = 1024
    for s, (pix, N, plane) in enumerate(cases):
        rows = pix.numel()
        want_crow, want_cpix, want_slot = _expect(pix, min(N, rows), rows, slot_init[s])
        nl = want_cpix.numel()
        assert int(nv[s]) == nl, (s, int(nv[s]), nl)
        cw, cv = crow[s]
        assert torch.equal(cv.cpu(), want_crow)
        pw, pv = cpix[s]
        assert torch.equal(pv[:nl].cpu(), want_cpix)
        assert bool((pv[nl:] == _GUARD).all()), "cpix written past n_local"
        for w in (cw, pw):
            assert bool((w[:g] == _GUARD).all()) and bool((w[-g:] == _GUARD).all()), "guard region written"
        if slots[s] is not None:
            sw, sv = slots[s]
            assert torch.equal(sv.cpu(), want_slot)
            assert bool((sw[:g] == _GUARD).all()) and bool((sw[-g:] == _GUARD).all())
        assert torch.equal(pix_d[s], before[id(pix_d[s])]) and torch.equal(n_d[s], before[id(n_d[s])])
    assert bool((nw[:g] == _GUARD).all()) and bool((nw[-g:] == _GUARD).all())
    return [int(x) for x in nv.cpu()]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["all", "none", "blocks", "single", "zero", "stale"])
def test_local_rows_one_scale(kind, dev):
    gen = torch.Generator().manual_seed(3)
    pix, N = _case(kind, 3000, 40000, gen)
    counts = _run_local_rows([(pix, N, 40000)], dev, with_slot=True)
    assert counts[0] == {"all": 3000, "none": 0, "single": 1, "zero": 0}.get(kind, counts[0])


@pytest.mark.gpu
def test_local_rows_upper_bound_and_many_scales(dev):
    """N at its upper bound (65 536 rows, 64 chunks of the CTA), row counts that are not a multiple of 32 or 1024,
    eight scales in one launch, with and without slot maps (half of the scales have one)."""
    gen = torch.Generator().manual_seed(5)
    cases = []
    for kind, rows in [("blocks", 65536), ("all", 1), ("single", 33), ("stale", 1025), ("none", 7), ("zero", 100),
                       ("blocks", 4097), ("all", 65536)]:
        pix, N = _case(kind, rows, 2 * 65536, gen)
        cases.append((pix, N, 2 * 65536))
    counts = _run_local_rows(cases, dev, with_slot=True)
    assert counts[1] == 1 and counts[7] == 65536 and counts[4] == 0
    _run_local_rows(cases[:3], dev, with_slot=False)


@pytest.mark.gpu
def test_local_rows_device_count_above_bound_is_clamped(dev):
    """A device count above `rows` is read as `rows`: nothing is read or written past the bound."""
    gen = torch.Generator().manual_seed(7)
    pix, _ = _case("all", 500, 1000, gen)
    _run_local_rows([(pix, 10 ** 6, 1000)], dev, with_slot=True)


# ---- 2. the pooled tail against the single-process tail on the concatenated batch -----------------------------------
def _inputs(n, dev, dtype, layout):
    from mscs_b200 import synth
    labels = synth.synth_labels(n, 128, 256, 19, 7, 16, 0.05, 21)
    zs = synth.synth_features(n, C_PREV, 128, 256, [4, 8, 16], 22)
    fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
    return labels.to(dev), [z.to(dev, dtype).contiguous(memory_format=fmt) for z in zs]


def _module(cfg, dev, comm=None):
    from mscs_b200 import ProjectorTailContrastive_ms
    torch.manual_seed(11)            # the same tails on every rank and in the single process
    return ProjectorTailContrastive_ms(dict(cfg), C_PREV, D, comm=comm).to(dev)


def _params(mod):
    return [t.weight for t in mod.tails] + [t.bias for t in mod.tails]


def _samples(mod):
    return [(s.pix.clone(), s.pair_ref.clone(), s.idx_ref.clone()) for s in mod.last_samples]


def _pooled(cfg, labels, zs, world, seed, dev, calls=2, second_backward=False):
    """`world` ranks on this GPU, rank r passing images [r nl, (r+1) nl); `calls` forward + backward steps each.
    Per rank, per call: loss, terms, samples and the gradients (z..., W..., b...)."""
    from mscs_b200 import _lib, _ops, projector
    nl = labels.shape[0] // world
    shared = _ops.ThreadComm._Shared(world)
    results, errors = [None] * world, []
    mods = [_module(cfg, dev, _ops.ThreadComm(shared, r)) for r in range(world)]     # (before the generator is seeded)

    def worker(r):
        try:
            torch.cuda.set_device(dev)
            mod = mods[r]
            lab = labels[r * nl:(r + 1) * nl]
            fts = [z[r * nl:(r + 1) * nl].detach().requires_grad_(True) for z in zs]
            S = len(fts)
            recs = []
            for _ in range(calls):
                loss = mod(lab, fts)
                st = mod.last_state
                Ws = [t.weight for t in mod.tails]
                dtypes = [f.dtype for f in fts] + [p.dtype for p in _params(mod)]
                if world == 1:      # a one-rank comm takes the single-process path (one thread: autograd is fine)
                    g = torch.autograd.grad(loss, fts + _params(mod))
                    gz, gW, gb, again = g[:S], g[S:2 * S], g[2 * S:], None
                else:
                    bwd = lambda: projector._backward_pooled(_lib.load(), st, torch.ones((), device=dev), Ws,
                                                             [True] * (3 * S), dtypes)
                    with torch.cuda.device(dev), _ops._pin_stream():
                        gz, gW, gb = bwd()
                        again = bwd() if second_backward else None
                torch.cuda.synchronize()
                recs.append(dict(loss=float(loss.detach()), grads=list(gz) + list(gW) + list(gb),
                                 again=(list(again[0]) + list(again[1]) + list(again[2])) if again else None,
                                 samples=_samples(mod),
                                 terms=[float(x) for x in mod.ms_losses] + [float(x) for x in mod.cs_losses]))
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


def _single(cfg, labels, zs, seed, dev, calls=2):
    mod = _module(cfg, dev)
    leaves = [z.detach().requires_grad_(True) for z in zs]
    torch.manual_seed(seed)
    recs = []
    for _ in range(calls):
        loss = mod(labels, leaves)
        grads = torch.autograd.grad(loss, leaves + _params(mod))
        recs.append(dict(loss=float(loss.detach()), grads=list(grads), samples=_samples(mod),
                         terms=[float(x) for x in mod.ms_losses] + [float(x) for x in mod.cs_losses]))
    return recs


def _cosine(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / torch.sqrt((a @ a) * (b @ b)))


def _matches_single(recs, single, zs, nl, planes):
    S = len(planes)
    want = single["loss"]
    for s, plane in enumerate(planes):          # sampling: exactly, every row sampled by one rank
        pix1, pair1, idx1 = single["samples"][s]
        owner = torch.zeros_like(pix1)
        for r, rec in enumerate(recs):
            pix, pair, idx = rec["samples"][s]
            assert torch.equal(pair, pair1)
            mine = pix >= 0
            owner += mine.int()
            assert torch.equal(pix[mine] + r * nl * plane, pix1[mine])
            own = (pair[:, 0] >= r * nl) & (pair[:, 0] < (r + 1) * nl)
            assert torch.equal(idx[own], idx1[own])
        assert bool((owner == 1).all())
    for r, rec in enumerate(recs):
        assert abs(rec["loss"] - want) < 2e-5 * abs(want), (r, rec["loss"], want)
        for a, b in zip(rec["terms"], single["terms"]):
            assert abs(a - b) < 2e-5 * abs(b)
        for s in range(S):
            g, w, z = rec["grads"][s], single["grads"][s][r * nl:(r + 1) * nl], zs[s][r * nl:(r + 1) * nl]
            assert g.dtype == z.dtype and g.shape == z.shape and g.stride() == z.stride()
            assert torch.equal((g != 0).any(dim=1), (w != 0).any(dim=1)), f"rank {r} scale {s}: sampled pixels differ"
            assert _cosine(g, w) > 0.99999, (r, s, _cosine(g, w))
    for j in range(S, 3 * S):                   # weights and biases: the ranks' contributions sum to the gradient
        tot = sum(rec["grads"][j].double() for rec in recs)
        ref = single["grads"][j].double()
        assert float((tot - ref).abs().max()) <= 1e-3 * float(ref.abs().max()), j


@pytest.mark.gpu
@pytest.mark.parametrize("world,sampler,dtype,layout", [
    (1, "reference", "fp32", "nchw"),
    (2, "reference", "fp32", "nchw"), (2, "philox", "bf16", "channels_last"), (2, "reference", "fp16", "channels_last"),
    (3, "philox", "fp32", "channels_last"), (3, "reference", "bf16", "nchw"),
    (8, "reference", "fp32", "channels_last"), (8, "philox", "fp16", "nchw")])
def test_pooled_tail_matches_single_process(world, sampler, dtype, layout, dev):
    """Two consecutive steps (both slab parities; the second draws from the generator state or call index the first
    left), world 3 with uneven 128-row shards."""
    cfg = dict(CFG, sampler="philox", sampler_seed=99) if sampler == "philox" else CFG
    labels, zs = _inputs(2 * world if world < 8 else 8, dev, DTYPES[dtype], layout)
    nl = labels.shape[0] // world
    single = _single(cfg, labels, zs, 5, dev)
    assert single[0]["samples"][0][0].numel() > 256          # several row tiles, so the row ranges matter
    torch.manual_seed(5)
    before = torch.get_rng_state()
    res = _pooled(cfg, labels, zs, world, 5, dev)
    if sampler == "philox":
        assert torch.equal(torch.get_rng_state(), before), "the Philox sampler touched the torch CPU generator"
    planes = [z.shape[2] * z.shape[3] for z in zs]
    for k in range(2):
        _matches_single([res[r][k] for r in range(world)], single[k], zs, nl, planes)


@pytest.mark.gpu
def test_pooled_tail_second_backward(dev):
    """A second backward through the same graph gives the first one's gradients (fresh rows, fresh dense gradients)."""
    labels, zs = _inputs(4, dev, torch.float32, "channels_last")
    for layout_zs in (zs, [z.contiguous() for z in zs]):
        res = _pooled(CFG, labels, layout_zs, 2, 5, dev, calls=1, second_backward=True)
        for r in range(2):
            rec = res[r][0]
            for g, h in zip(rec["grads"], rec["again"]):
                assert g.stride() == h.stride()
                assert float((g.double() - h.double()).abs().max()) <= 1e-3 * float(g.double().abs().max())


@pytest.mark.gpu
def test_pooled_tail_refusals(dev):
    import mscs_b200
    from mscs_b200 import _ops, synth
    # CUDA-graph capture of the pooled mode: refused before anything is enqueued
    cfg = dict(CFG, sampler="philox", sampler_seed=1)
    mod = _module(cfg, dev, _ops.ThreadComm(_ops.ThreadComm._Shared(2), 0))
    labels, zs = _inputs(2, dev, torch.float32, "nchw")
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="pooled mode"):
        with torch.cuda.graph(g):
            mod(labels[:1], [z[:1] for z in zs])
    torch.cuda.synchronize()
    assert float(torch.ones(4, device=dev).sum()) == 4.0
    # NCHW planes that are not a multiple of 8 pixels
    lab = synth.synth_labels(2, 60, 100, 19, 6, 4, 0.05, 3).to(dev)
    z = synth.synth_features(2, C_PREV, 60, 100, [4], 4)[0].to(dev)     # 15 x 25 plane
    one = dict(CFG, scales=1, weights=[1.0], cross_scale_contrast=False)
    mod = mscs_b200.ProjectorTailContrastive_ms(one, C_PREV, D, comm=_ops.ThreadComm(_ops.ThreadComm._Shared(2), 0))
    with pytest.raises(NotImplementedError, match="multiple of 8"):
        mod.to(dev)(lab[:1], [z[:1]])


# ---- no device: argument checks ---------------------------------------------------------------------------------
def _call(count=1, pix=_FAKE, n_rows_dev=_FAKE, rows=10, crow=_FAKE, cpix=_FAKE, slot=None, n_local=_FAKE):
    import mscs_b200
    from mscs_b200 import _lib
    lib = mscs_b200.load()
    k = max(count, 1)
    arr = lambda p: _lib.ptr_array([p] * k)
    rc = lib.mscs_local_rows_batch(arr(pix), arr(n_rows_dev), (C.c_int32 * k)(*([rows] * k)), arr(crow), arr(cpix),
                                   arr(slot) if slot is not None else None, n_local, count, None)
    return rc, lib.mscs_last_error()


def test_local_rows_rejects_bad_arguments():
    for kw, what in [(dict(count=0), b"count"), (dict(count=9), b"count"), (dict(pix=None), b"null"),
                     (dict(n_rows_dev=None), b"null"), (dict(crow=None), b"null"), (dict(cpix=None), b"null"),
                     (dict(n_local=None), b"null"), (dict(rows=-1), b"rows"), (dict(pix=_FAKE + 2), b"aligned"),
                     (dict(crow=_FAKE + 1), b"aligned"), (dict(slot=_FAKE + 2), b"aligned"),
                     (dict(n_local=_FAKE + 2), b"aligned"), (dict(n_rows_dev=_FAKE + 3), b"aligned")]:
        rc, msg = _call(**kw)
        assert rc < 0 and what in msg, (kw, rc, msg)

