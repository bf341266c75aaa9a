"""Projector tail evaluated on the SAMPLED rows only (SURVEY.md section 8f, item 1).

The reference's projector (models/Projector.py:49-72) ends in ``nn.Conv2d(c_prev, d, kernel_size=1)``: a d x c_prev
matrix applied to every pixel of every scale (HRNet.py:642, UPerNet.py:241), although the contrastive loss reads at most
``max_features_total`` pixels per scale -- at the HRNet-W48 Cityscapes shape 32 604 of 522 240 pixels (6 %).  This module
takes the feature maps in front of that last convolution and evaluates

    DenseContrastiveLossV2_ms(config)(label, [conv_s(z_s) for s])          (losses/DenseContrastiveLossV2_ms.py:44-82)

without ever forming the dense projector output or its dense gradient, in the device-driven order of the drop-in classes
(one host wait per forward, none under CUDA-graph capture):

    fills; K1 sampling on the high-priority stream (plan records fetched behind it)    -> slot maps / pixel ids per row
    raw gather of the sampled c_prev-vectors (mscs_gather_raw[_rows]_batch)          Z_s  (Ncap_s, c_prev), maps read
                                                                                      in their own dtype and layout
    P_s = Z_s W_s^T + b_s                                                            library GEMM, fp32, autocast off
    row normalisation -> bf16 operands (mscs_gather_rows_nhwc_batch on the rows of P, device row counts)
    K3 with device row counts; then the plan records reach the host
    backward: K4, normalisation backward -> dP_s;  dZ_s = dP_s W_s, dW_s = dP_s^T Z_s, db_s = sum dP_s
    raw dense writer of dZ_s into the gradient of z_s, in z_s's dtype and memory format

The GEMMs run over the upper bound Ncap_s = min(max_features_total, n h w) of the rows, so that eager and captured
calls are the same work; rows at and above the call's count N_s of Z_s and dP_s are cleared on every call, which keeps
dW_s and db_s exact.  Same loss, same gradients w.r.t. z_s, W_s and b_s as the dense evaluation
(tests/test_gpu_projector.py, tests/test_gpu_projector_tail.py).  It is NOT a reference class name: the reference has no
such module, so it sits next to the drop-in classes with its own, explicit interface.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib, _ops
from .datasets import class_facts
from .losses import _GraphReadout, _fetch_logged, _philox_key, _spec_from_config


def _al(x):
    return (x + 63) // 64 * 64          # 256-byte aligned fp32 regions (GEMM operands, row kernels)


class _TailWorkspace(_ops._Workspace):
    """The drop-in's workspace of the loss on the projected rows (sampling, operand matrices, row statistics, gradient
    accumulators), plus the rows of the tail: Z (Ncap x c_prev), P and dP (Ncap x d) per scale, with every ctypes item
    that depends only on their addresses built once."""

    def __init__(self, sp, c_prev, graph=False):
        super().__init__(sp, graph)
        dev, S, d = sp.dev, sp.S, sp.C
        f32 = torch.float32
        zn = [_al(sp.Ncap[s] * c_prev[s]) for s in range(S)]
        pn = [_al(sp.Ncap[s] * d) for s in range(S)]
        # Z and dP in one slab: cleared by the same fill, on every call
        self.zd = torch.empty(sum(zn) + sum(pn), dtype=f32, device=dev)
        self.P = torch.empty(sum(pn), dtype=f32, device=dev)
        self.Z, self.dP, self.Pr, zo, po = [], [], [], 0, 0
        for s in range(S):
            N = sp.Ncap[s]
            self.Z.append(self.zd[zo:zo + N * c_prev[s]].view(N, c_prev[s]))
            self.dP.append(self.zd[sum(zn) + po:sum(zn) + po + N * d].view(N, d))
            self.Pr.append(self.P[po:po + N * d].view(N, d))
            zo += zn[s]
            po += pn[s]
        self.iota = torch.arange(max(sp.Ncap), dtype=torch.int32, device=dev)      # the rows of P are the anchor rows
        self.tail_fill = (_lib.ptr_array([self.dF_ptr, self.zd.data_ptr()]), (C.c_int32 * 2)(0, 0),
                          (C.c_size_t * 2)(4 * sp.dF_n, 4 * self.zd.numel()))
        fb = self.fbase
        pix = [self.islab.data_ptr() + 4 * sp.ioff[s][2] for s in range(S)]
        self.pitems, self.nitems = (_lib.RowsItem * S)(), (_lib.RowsItem * S)()
        self.raw = (_lib.RowsItem * S)() if sp.nhwc else (_lib.GatherItem * S)()
        for s in range(S):
            n, _d, h, w = sp.feat_shapes[s]
            for it in (self.pitems[s], self.nitems[s]):         # normalisation of the rows of P, and its backward
                it.pix, it.n_rows_dev, it.rows, it.C = self.iota.data_ptr(), self.rows_dev[s], sp.Ncap[s], d
                it.anc_f32, it.inv_norm = fb + 4 * sp.foff[s][0], fb + 4 * sp.foff[s][1]
            self.pitems[s].feat, self.pitems[s].anc_bf16 = self.Pr[s].data_ptr(), self.bbase + 2 * sp.boff[s]
            it = self.nitems[s]
            it.dF, it.ldF, it.dfeat = self.dF_ptr + 4 * sp.dF_off[s], sp.C_pad, self.dP[s].data_ptr()
            it = self.raw[s]
            if sp.nhwc:
                it.pix, it.n_rows_dev, it.rows = pix[s], self.rows_dev[s], sp.Ncap[s]
            else:
                it.n, it.plane, it.slot = n, h * w, self.slots[s].data_ptr()
            it.C, it.anc_f32 = c_prev[s], self.Z[s].data_ptr()
        self.pix = pix


class _ProjTailFn(torch.autograd.Function):
    """(labels, spec, holder, S, z_0..z_{S-1}, W_0..W_{S-1}, b_0..b_{S-1}) -> (total 0-d, term losses)."""

    @staticmethod
    def forward(ctx, labels, spec, holder, S, *tensors):
        lib = _lib.load()
        zs, Ws, bs = tensors[:S], tensors[S:2 * S], tensors[2 * S:3 * S]
        plans, philox = holder["plans"], holder.get("philox")
        d = Ws[0].shape[0]
        key = lambda nhwc: (zs[0].device, tuple(labels.shape), tuple(tuple(z.shape) for z in zs), d, nhwc)
        # decided (and refused) before anything is enqueued
        graph = _ops.graph_mode(spec, 1, False, labels, zs, philox[1] if philox is not None else None,
                                plan_of=lambda nhwc: plans.get(key(nhwc)))
        dev = zs[0].device
        for t in tensors:
            _ops._require_device(t)
        if not lib.mscs_device_ok():
            raise RuntimeError("mscs_b200 needs a compute-capability 10.x (B200) device; no fallback exists")
        nhwc = _ops.channels_last_ok(spec, 1, zs)
        if not nhwc and any((z.shape[2] * z.shape[3]) % 8 for z in zs):
            raise NotImplementedError("the projector-tail path needs feature planes that are a multiple of 8 pixels "
                                      "(or channels-last maps)")
        labels = labels.to(dev)
        if labels.dtype != torch.int64:
            labels = labels.long()
        labels = labels.contiguous()
        needs = [bool(x) for x in ctx.needs_input_grad[4:]]
        c_prev = [W.shape[1] for W in Ws]
        maps = []
        for z in zs:                # read as they are: fp32, bf16, fp16 (anything else as an fp32 copy)
            m = z.detach()
            if m.dtype not in _ops._DTYPE_CODE:
                m = m.float()
            maps.append(m if nhwc else m.contiguous())
        with torch.cuda.device(dev), _ops._pin_stream():
            sp = plans.get(key(nhwc))
            if sp is None:
                sp = plans[key(nhwc)] = _ops._StepPlan(dev, labels.shape, [(z.shape[0], d, z.shape[2], z.shape[3])
                                                                           for z in zs], spec, False, nhwc=nhwc)
            state, total = _forward(lib, sp, labels, maps, Ws, bs, c_prev, needs[:S], any(needs), philox, graph)
        holder["samples"], holder["state"] = state.samples, state
        ctx.state, ctx.S, ctx.needs = state, S, needs
        ctx.save_for_backward(*Ws)
        ctx.dtypes = [t.dtype for t in tensors]
        terms = state.term_loss
        ctx.mark_non_differentiable(terms)
        ctx.set_materialize_grads(False)
        return total, terms

    @staticmethod
    def backward(ctx, grad_total, _grad_terms):
        S = ctx.S
        if grad_total is None:
            return (None,) * (4 + 3 * S)
        with torch.cuda.device(ctx.state.sp.dev), _ops._pin_stream():
            gz, gW, gb = _backward(_lib.load(), ctx.state, grad_total, ctx.saved_tensors, ctx.needs, ctx.dtypes)
        return (None, None, None, None, *gz, *gW, *gb)


def _forward(lib, sp, labels, maps, Ws, bs, c_prev, needs_z, any_grad, philox, graph):
    """One forward in the device-driven order (module docstring).  graph: captured call, nothing waits for the host."""
    dev, S, A = sp.dev, sp.S, sp.A
    st, cur = _ops._stream(), _ops._cur_stream()
    e = _TailWorkspace(sp, c_prev, graph=True) if graph else (sp.ws_pool.pop() if sp.ws_pool else _TailWorkspace(sp, c_prev))
    if e.last_stream is not None and e.last_stream != cur:
        cur.wait_stream(e.last_stream)          # reuse on another stream: order after its previous user
    e.last_stream = cur
    nt = len(sp.terms)
    out = torch.empty(nt + 2, dtype=torch.float32, device=dev)      # term losses, total, inf/NaN flag
    total_t = torch.empty((), dtype=torch.float32, device=dev)      # own buffer, not a view (see _ops._run_forward_fast)
    for job in (e.job_fwd, e.job_bwd):
        job.term_loss, job.total_loss = out.data_ptr(), out.data_ptr() + 4 * nt
        job.total_out = total_t.data_ptr()
    hp = _ops._hp_stream(dev) if _ops._USE_HP_STREAM else None
    ss = hp if hp is not None else cur
    st_s = C.c_void_p(ss.cuda_stream)
    if hp is not None:
        hp.wait_stream(cur)
    if philox is None:          # MT19937 stream of the torch CPU generator (normally produced during the previous step)
        mt, pos = _ops.torch_mt_state()
        cache = _ops._stream_cache(dev)
        draws = cache.acquire_nowait(mt, pos, sp.max_draws + _ops._MT_N).data_ptr()
        ss.wait_event(cache.ready)
    else:
        if e.philox is None:
            e.philox = torch.empty((sp.max_draws + 3) // 4 * 4 + 4, dtype=torch.int32, device=dev)
        draws = e.philox.data_ptr()
        if graph:
            _lib.check(lib.mscs_philox_stream_dev(int(philox[0]) & (2 ** 64 - 1), philox[1].data_ptr(), sp.max_draws,
                                                  draws, st_s), "mscs_philox_stream_dev")
        else:
            _lib.check(lib.mscs_philox_stream(int(philox[0]) & (2 ** 64 - 1), int(philox[1]), sp.max_draws, draws,
                                              st_s), "mscs_philox_stream")
    # channels-last dense gradients: pre-zeroed on a side stream, the sampled rows stored by the backward
    gradbufs = _ops._GradBuffers(maps, needs_z, True, 0) if (sp.nhwc and any(needs_z)) else None
    if gradbufs is not None:
        if graph:       # filled on the caller's stream: a forward captured without its backward leaves no open fork
            gradbufs.side = cur
        gradbufs.start_fill()
    # main stream, next to the sampling chain: gradient-row accumulators, Z and dP
    _lib.check(lib.mscs_fill_bytes(*e.tail_fill, 2, st), "mscs_fill_bytes")
    # sampling stream: statistics / slot-map fills, plan, plan records to the host, selection from the device records
    _lib.check(lib.mscs_fill_bytes(e.fill_ptrs, e.fill_vals, e.fill_bytes, 2, st_s), "mscs_fill_bytes")
    fn, fname = _ops._plan_entry(lib, labels)
    _lib.check(fn(C.byref(sp.cfg), labels.data_ptr(), e.ws, e.plan_dev, st_s), fname)
    if not graph:
        _lib.check(lib.mscs_plan_fetch_begin(e.plan_dev, S, st_s), "mscs_plan_fetch_begin")
    _lib.check(lib.mscs_sample_select_async(C.byref(sp.cfg), e.plan_dev, sp.v_cap, e.ws, draws, *e.arrs, e.sarr, st_s),
               "mscs_sample_select_async")
    if hp is not None:
        cur.wait_stream(hp)
    for s in range(S):
        e.raw[s].feat, e.raw[s].dtype = maps[s].data_ptr(), _ops._DTYPE_CODE[maps[s].dtype]
    if sp.nhwc:
        _lib.check(lib.mscs_gather_raw_rows_batch(e.raw, S, st), "mscs_gather_raw_rows_batch")
    else:
        _lib.check(lib.mscs_gather_raw_batch(e.raw, S, st), "mscs_gather_raw_batch")
    with torch.autocast("cuda", enabled=False):     # the 1x1 convolution of the sampled pixels, fp32 as nn.Conv2d
        for s in range(S):
            W = Ws[s].detach().float().reshape(sp.C, c_prev[s])
            torch.addmm(bs[s].detach().float(), e.Z[s], W.t(), out=e.Pr[s])
    _lib.check(lib.mscs_gather_rows_nhwc_batch(e.pitems, S, st), "mscs_gather_rows_nhwc_batch")
    _lib.check(lib.mscs_sim_forward(C.byref(e.job_fwd), st), "mscs_sim_forward")
    state = _ops._StepState()
    state.sp, state.entry, state.graph = sp, e, graph     # (from here on an exception returns the workspace to the pool)
    state.samples = None
    if not graph:
        plan = e.plan
        _lib.check(lib.mscs_plan_fetch_end(plan, S), "mscs_plan_fetch_end")       # the one host wait
        _ops._raise_plan_errors(plan, S, sp.spec)
        state.samples = [_ops.ScaleSample(plan[s].T, plan[s].V, plan[s].N, bool(plan[s].log_flag), plan[s].dl_h,
                                          plan[s].dl_w, e.islab, sp.ioff[s], A) for s in range(S)]
        for i, (a, k, *_rest) in enumerate(sp.terms):      # the eager backward is launched with the actual counts
            t = e.job_bwd.terms[i]
            t.N1, t.N2 = state.samples[a].N, state.samples[k].N
        if philox is None:
            _ops._finish_rng(sp, dev, mt, pos, sum(int(plan[s].draws) for s in range(S)), defer=any_grad)
    state.job, state.gradbufs = e.job_bwd, gradbufs
    state.scalars, state.term_loss = out, out[:nt]
    state.num_ms, state.cs_logged, state.comm = S, sp.cs_logged, None
    # the 0-d loss is not kept by the state: an output of the Function references its grad_fn, which owns the state
    return state, total_t


def _backward(lib, state, grad_total, Ws, needs, dtypes):
    sp, e = state.sp, state.entry
    dev, S = sp.dev, sp.S
    st, cur = _ops._stream(), _ops._cur_stream()
    if getattr(state, "bwd_done", False):       # a second backward through the same graph: fresh accumulators
        _lib.check(lib.mscs_fill_bytes(e.tail_fill[0], e.tail_fill[1], e.tail_fill[2], 1, st), "mscs_fill_bytes")
    state.bwd_done = True
    g = grad_total.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
    _lib.check(lib.mscs_sim_backward(C.byref(state.job), g.data_ptr(), e.bw_ptrs, e.bw_lds, st), "mscs_sim_backward")
    if not state.graph:
        _ops._stream_cache(dev).flush()        # the deferred generator launch of the next call's stream
    _lib.check(lib.mscs_scatter_rows_nhwc_batch(e.nitems, S, st), "mscs_scatter_rows_nhwc_batch")      # normalise^T
    gz, gW, gb, dZ = [None] * S, [None] * S, [None] * S, {}
    with torch.autocast("cuda", enabled=False):
        for s in range(S):
            W = Ws[s].detach().float().reshape(sp.C, -1)
            if needs[s]:
                dZ[s] = e.dP[s] @ W                                                       # (Ncap, c_prev)
            if needs[S + s]:
                gW[s] = (e.dP[s].t() @ e.Z[s]).reshape(Ws[s].shape).to(dtypes[S + s])
            if needs[2 * S + s]:
                gb[s] = e.dP[s].sum(0).to(dtypes[2 * S + s])
    idx = sorted(dZ)
    if not idx:
        return gz, gW, gb
    io = [dt if dt in _ops._DTYPE_CODE else torch.float32 for dt in dtypes[:S]]      # dtypes the kernels write
    if sp.nhwc:         # raw row stores into the pre-zeroed channels-last gradients
        gbuf = state.gradbufs
        if gbuf is not None:
            cur.wait_event(gbuf.ready)
        items = (_lib.RowsItem * len(idx))()
        for j, s in enumerate(idx):
            n, c, h, w = sp.feat_shapes[s][0], dZ[s].shape[1], sp.feat_shapes[s][2], sp.feat_shapes[s][3]
            buf = gbuf.take(s) if gbuf is not None else None
            if buf is None:      # second backward through the same graph
                buf = torch.zeros((n, h, w, c), dtype=io[s], device=dev).permute(0, 3, 1, 2)
            gz[s] = buf
            it = items[j]
            it.pix, it.n_rows_dev, it.rows, it.C = e.pix[s], e.rows_dev[s], sp.Ncap[s], c
            it.dF, it.ldF, it.dfeat, it.dtype = dZ[s].data_ptr(), c, buf.data_ptr(), _ops._DTYPE_CODE[io[s]]
        _lib.check(lib.mscs_scatter_rows_nhwc_batch(items, len(idx), st), "mscs_scatter_rows_nhwc_batch")
    else:               # NCHW: every byte of the gradients written once, the sampled pixels from the rows dZ
        shapes = [(sp.feat_shapes[s][0], dZ[s].shape[1], sp.feat_shapes[s][2], sp.feat_shapes[s][3]) for s in idx]
        _slab, views, offs = _ops._dense_grad_slab(shapes, [io[s] for s in idx], dev)
        items, rows = (_lib.ScatterItem * len(idx))(), (C.c_int32 * len(idx))()
        for j, s in enumerate(idx):
            n, c, h, w = shapes[j]
            gz[s] = views[j]
            it = items[j]
            it.dF, it.ldF, it.slot, it.n, it.C, it.plane = dZ[s].data_ptr(), c, e.slots[s].data_ptr(), n, c, h * w
            it.dfeat, it.dtype = views[j].data_ptr(), _ops._DTYPE_CODE[io[s]]
            rows[j] = sp.Ncap[s]
        _lib.check(lib.mscs_scatter_dense_batch(items, rows, len(idx), st), "mscs_scatter_dense_batch")
    for s in idx:
        if gz[s].dtype != dtypes[s]:
            gz[s] = gz[s].to(dtypes[s])
    return gz, gW, gb


class ProjectorTailContrastive_ms(_GraphReadout, nn.Module):
    """``forward(label, pre_features)`` == ``DenseContrastiveLossV2_ms(config)(label, [tail_s(z_s) for s])`` with
    ``tail_s = nn.Conv2d(c_prev_s, d, 1)`` -- the LAST layer of the reference's projector (Projector.py:69), owned by
    this module as ``self.tails[s]`` (``from_projector`` takes them out of a reference ``Projector``).

    Same config keys as DenseContrastiveLossV2_ms (losses.py), ``sampler='philox'`` included; exposes ``ms_losses`` /
    ``cs_losses`` / ``cross_scale_contrast`` like it, so the reference's logger reads it the same way, and the same
    readout (``fetch_logged``, ``fetch_samples``, ``nan_flag``, ``graph_call_index``) for CUDA-graph capture.  The maps
    z_s may be fp32, bf16 or fp16, NCHW or channels-last; their gradients come back in the same dtype and layout."""

    def __init__(self, config, c_prev, d=256):
        super().__init__()
        self.scales = config["scales"] if "scales" in config else 2
        self.weights = config["weights"] if "weights" in config else [1.0] * self.scales
        assert self.scales == len(self.weights)
        c_prev = [c_prev] * self.scales if isinstance(c_prev, int) else list(c_prev)
        assert len(c_prev) == self.scales
        self.num_all_classes = class_facts(config["dataset"], config["experiment"])[0]
        self._spec = _spec_from_config(config, self.scales, self.weights, ms=True)
        self.cross_scale_contrast = self._spec.cross_scale
        self.tails = nn.ModuleList([nn.Conv2d(c, d, kernel_size=1, stride=1) for c in c_prev])
        self.ms_losses, self.cs_losses = [], []
        self.log_this_step = False
        self.last_samples = None
        self._sampler_calls = 0
        self._plans = {}            # step plans of the input shapes seen so far (their workspaces are pooled there)

    @classmethod
    def from_projector(cls, config, projector):
        """Takes over the final 1x1 convolution of every ``project{i}`` of a reference ``Projector`` (is_ms) and
        returns ``(module, bodies)`` with ``bodies[i]`` = that Sequential without its last layer."""
        names = [f"project{i}" for i in range(len(projector.c_in))] if projector.is_ms else ["project"]
        seqs = [getattr(projector, nm) for nm in names]
        lasts = [seq[-1] for seq in seqs]
        mod = cls(config, [l.in_channels for l in lasts], lasts[0].out_channels)
        for mine, theirs in zip(mod.tails, lasts):
            mine.load_state_dict(theirs.state_dict())
        return mod, [nn.Sequential(*list(seq.children())[:-1]) for seq in seqs]

    def forward(self, label, pre_features):
        feats = list(pre_features[:self.scales])
        if len(feats) < self.scales:
            raise IndexError("list index out of range")
        holder = {"plans": self._plans}
        _philox_key(self, holder, feats[0].device)
        total, terms = _ProjTailFn.apply(label, self._spec, holder, self.scales, *feats,
                                         *[t.weight for t in self.tails], *[t.bias for t in self.tails])
        state = holder["state"]
        self.last_samples, self.last_state = holder["samples"], state
        self.ms_losses = [terms[s] for s in range(state.num_ms)]
        self.cs_losses = [terms[i] for i in state.cs_logged]
        self.nan_flag = state.scalars[-1]                # 0-d device tensor: 1.0 if the loss is inf/NaN (no sync)
        if holder["samples"] is not None and any(s.log_flag for s in holder["samples"]):
            self.log_this_step = True
        return total

    def fetch_logged(self, state=None):
        """Scalars of the last call (or of ``state``) for the logger in one device->host copy, as
        ``DenseContrastiveLossV2_ms.fetch_logged`` (a captured call: its latest replay)."""
        st = self.last_state if state is None else state
        return _fetch_logged(self, st, st.num_ms, st.cs_logged)
