"""Host orchestration of the CUDA path and the single ``torch.autograd.Function`` on top of it.

PyTorch is plumbing here (device memory from the caching allocator, the current stream, autograd
bookkeeping); every computation between "labels + feature maps in" and "scalar loss / dense
feature gradients out" is a libmscs.so kernel.  Nothing in this module computes on the CPU and
there is no fallback: a missing library or a non-sm_100 device raises.
"""
import ctypes as C
import os
import struct
import threading
from dataclasses import dataclass, field
from typing import List

import numpy as np
import torch

from . import _lib

_MT_N = 624
# tuning switch, read once at import (nothing on the per-step path calls getenv)
_USE_HP_STREAM = os.environ.get("MSCS_HP", "1") != "0"       # sampling kernels on a high-priority stream
# NCHW dense gradients are written in ONE streaming pass by the backward (k_dense_stream); bench.py reads this flag
_DENSE_ONE_PASS = True
# element types the kernels read and write natively (MSCS_DTYPE_* codes of the C ABI); see half_io_ok
_DTYPE_CODE = {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16}

# optional per-stage device timing (bench.py): {stage: [(start_event, end_event), ...]} or None
TIMING = None
# stage accounting level: True = every stage (16 extra event records per step: ~50 us of step time at cfg-2, the
# records also sit between kernels that otherwise overlap through programmatic dependent launch); False = only the
# dominant kernel (`sim_bwd`, 2 events) -- what bench.py uses inside its timed region
TIMING_ALL = True
# optional host-side accounting (tools/stage_times.py): seconds the host spent blocked in the plan fetch, per call
HOST_WAIT = None
# optional host-side segment accounting (tools/stage_times.py): {segment: seconds}
HOST_SEG = None


def _seg(name, t0):
    """Adds the host time since t0 to segment `name`; returns the new time stamp (no-op when disabled)."""
    if HOST_SEG is None:
        return t0
    import time
    t1 = time.perf_counter()
    HOST_SEG[name] = HOST_SEG.get(name, 0.0) + (t1 - t0)
    return t1


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        self.on = TIMING is not None and (TIMING_ALL or self.name == "sim_bwd")
        if self.on:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *exc):
        if self.on:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            TIMING.setdefault(self.name, []).append((self.e0, e1))


def LAUNCHES_PER_STEP(num_scales, single_scale):
    """Kernels of libmscs.so launched by one forward+backward (torch fills not counted; checked against the ncu
    launch list in profiles/): K1 hist, tile-scan, plan, MT19937 stream, select (5); K2 (1); K3 row ranges,
    work tables of both sweeps (one launch), 2 sweeps, finalise (5); K4 work table + backward (2);
    normalisation backward of the rows + one-pass dense writer (2)."""
    return 5 + 1 + 5 + 2 + 2      # gather and scatter: one launch each for all scales


@dataclass
class LossSpec:
    """Flat, resolved loss configuration (see losses.py for the reference key rules)."""
    num_classes: int
    temperature: float
    cs_temperature: float
    min_views: int = 5
    max_views: int = 2500
    max_total: int = 10000
    weights: List[float] = field(default_factory=lambda: [1.0])
    cross_scale: bool = False
    detach_deepest: bool = False
    w_high_low: float = 1.0
    w_high_mid: float = 1.0
    # not reference keys: "reference" = the torch CPU generator consumed exactly like the reference's randperm calls;
    # "philox" = opt-in counter-based stream keyed by (sampler_seed, call index) (SURVEY.md 8f item 4)
    sampler: str = "reference"
    seed: int = 0


class ScaleSample:
    """Sampling result of one scale.  The arrays live in one int32 slab; views are made on demand.

      idx_ref  (T, V) int32  flat pixel index in REFERENCE order (V2.py:122)
      pair_ref (T, 2) int32  (image, class) in reference order (V2.py:106-107)
      pix (N,) int32 image*plane + pixel, rows sorted by class;  cls (N,) class of each sorted row
      seg (A+1,) int32 class segments of the sorted rows
    """
    __slots__ = ("T", "V", "N", "log_flag", "dl_h", "dl_w", "_slab", "_off", "_A")

    def __init__(self, T, V, N, log_flag, dl_h, dl_w, slab, off, A):
        self.T, self.V, self.N, self.log_flag, self.dl_h, self.dl_w = T, V, N, log_flag, dl_h, dl_w
        self._slab, self._off, self._A = slab, off, A

    def _view(self, k, n):
        return self._slab[self._off[k]:self._off[k] + n]

    idx_ref = property(lambda self: self._view(0, self.N).view(self.T, self.V))
    pair_ref = property(lambda self: self._view(1, 2 * self.T).view(self.T, 2))
    pix = property(lambda self: self._view(2, self.N))
    cls = property(lambda self: self._view(3, self.N))
    seg = property(lambda self: self._view(4, self._A + 1))

    def ptr(self, k):
        return self._slab.data_ptr() + 4 * self._off[k]


_stream_override = [None, None]


def _stream():
    """cudaStream_t of the current torch stream (looked up once per forward/backward call)."""
    if _stream_override[0] is not None:
        return _stream_override[0]
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _cur_stream():
    """torch Stream object of the current stream (cached for the duration of a forward/backward call:
    torch.cuda.current_stream() costs ~5 us of Python per call)."""
    if _stream_override[1] is not None:
        return _stream_override[1]
    return torch.cuda.current_stream()


class _pin_stream:
    def __enter__(self):
        cur = torch.cuda.current_stream()
        _stream_override[0], _stream_override[1] = C.c_void_p(cur.cuda_stream), cur

    def __exit__(self, *exc):
        _stream_override[0] = _stream_override[1] = None


class CompactLabels:
    """int16 label map produced by the fused label pass (csrc/ce.cu:k_label_pass; -1 = outside [0, A)): accepted by the
    loss classes in place of the int64 labels -- K1 then reads a quarter of the bytes, with identical results."""
    __slots__ = ("lab16", "hist", "shape", "num_classes")

    def __init__(self, lab16, hist, num_classes):
        self.lab16, self.hist, self.shape, self.num_classes = lab16, hist, tuple(lab16.shape), num_classes

    @property
    def device(self):
        return self.lab16.device


def _plan_entry(lib, labels, hist_only=False):
    """(function, name) of the K1 entry point for int64 or compact int16 labels."""
    i16 = labels.dtype == torch.int16
    if hist_only:
        return (lib.mscs_sample_hist_i16, "mscs_sample_hist_i16") if i16 else (lib.mscs_sample_hist, "mscs_sample_hist")
    return (lib.mscs_sample_plan_i16, "mscs_sample_plan_i16") if i16 else (lib.mscs_sample_plan, "mscs_sample_plan")


def _require_device(t):
    if not t.is_cuda:
        raise RuntimeError("mscs_b200 runs on a B200 GPU only: got a CPU tensor (there is no CPU fallback)")


# ---- torch CPU generator <-> MT19937 state ----------------------------------------------------
def torch_mt_state():
    """(state uint32[624], pos) of the torch CPU default generator (at::mt19937 layout:
    [seed u64][left i32][seeded i32][next u64][624 x u64] ...)."""
    raw = torch.get_rng_state().numpy()
    _last_raw[0] = raw
    _seed, left, _seeded, nxt = struct.unpack_from("<QiiQ", raw[:24].tobytes(), 0)
    mt = np.ascontiguousarray(raw[24:24 + 8 * _MT_N].view(np.uint64).astype(np.uint32))
    pos = _MT_N if left == 1 else int(nxt)
    return mt, pos


_last_raw = [None]      # serialised generator state read by the last torch_mt_state() (seed / header bytes are reused)


def _publish_mt_state(mt, pos):
    """Writes (state uint32[624], pos in 1..624) into the torch CPU default generator."""
    raw = _last_raw[0]
    raw = torch.get_rng_state().numpy().copy() if raw is None else raw.copy()
    _last_raw[0] = None
    hdr = struct.pack("<ii", 625 - pos, 1)
    raw[8:16] = np.frombuffer(hdr, dtype=np.uint8)
    raw[16:24] = np.frombuffer(struct.pack("<Q", pos), dtype=np.uint8)
    raw[24:24 + 8 * _MT_N] = mt.astype(np.uint64).view(np.uint8)
    torch.set_rng_state(torch.from_numpy(raw))


def torch_mt_advance(mt, pos, draws):
    """Advance the torch CPU default generator by ``draws`` 32-bit outputs -- what the reference's
    per-pair ``torch.randperm`` calls would have consumed (V2.py:121).  Returns the new (mt, pos)."""
    if draws <= 0:
        return mt, pos
    lib = _lib.load()
    mt = mt.copy()
    cpos = C.c_int(pos)
    _lib.check(lib.mscs_mt19937_advance_host(mt.ctypes.data_as(C.c_void_p), C.byref(cpos), C.c_uint64(draws)),
               "mscs_mt19937_advance_host")
    _publish_mt_state(mt, cpos.value)
    return mt, cpos.value


class _StreamCache:
    """MT19937 output streams produced ahead of time on a side CUDA stream.

    The stream a call needs depends only on the torch CPU generator state, and after a call that
    state is known (we advance it ourselves), so the next call's stream is generated while this
    call's tensor kernels run.  A call whose generator state is not the predicted one (first call,
    reseeding, another consumer of the generator) regenerates inline -- results are identical."""

    def __init__(self, dev):
        self.dev = dev
        self.side = torch.cuda.Stream(device=dev)
        self.bufs = [None, None]
        self.cur = 0
        self.key = None          # (state bytes, pos) the buffer `cur` was generated from
        self.words = 0
        self.ready = None        # event: buffer `cur` complete
        self.last_use = [None, None]   # event: last main-stream reader of each buffer
        self.lock = threading.Lock()
        self.pending = None      # deferred prefetch request (mt, pos, words), see release_and_prefetch
        self.host = [None, None]       # pinned host mirrors of the raw streams (see state_after)
        self.host_ready = None         # event: mirror of buffer `cur` complete
        self.copy = torch.cuda.Stream(device=dev)      # read-back of the generator state (see state_after)

    def _generate(self, which, mt, pos, words):
        lib = _lib.load()
        if self.bufs[which] is None or self.bufs[which].numel() < words + 1024:
            self.bufs[which] = torch.empty(words + 1024, dtype=torch.int32, device=self.dev)
            self.bufs[which].record_stream(self.side)
            self.side.wait_stream(_cur_stream())      # fresh allocation: order after its previous users
        # the stream depends only on the host-side generator state: it is NOT ordered after the main
        # stream, only after the last reader of this buffer (the selection kernel two calls ago)
        if self.last_use[which] is not None:
            self.side.wait_event(self.last_use[which])
        timed = TIMING is not None and TIMING_ALL
        if timed:          # stage accounting (bench.py): duration of the generator kernel on the side stream
            t0 = torch.cuda.Event(enable_timing=True)
            t0.record(self.side)
        _lib.check(lib.mscs_mt19937_stream(mt.ctypes.data_as(C.c_void_p), pos, C.c_uint64(words),
                                           self.bufs[which].data_ptr(), C.c_void_p(self.side.cuda_stream)),
                   "mscs_mt19937_stream")
        if timed:
            t1 = torch.cuda.Event(enable_timing=True)
            t1.record(self.side)
            TIMING.setdefault("mt_stream_side", []).append((t0, t1))
        ev = torch.cuda.Event()
        ev.record(self.side)
        # pinned host mirror of the raw stream, copied behind the generator on the side stream (2 MB at cfg-2): the
        # forward reads the next generator state out of it (state_after) without a device round trip in the window
        # between the plan fetch and the launch of the backward
        hb = self.host[which]
        if hb is None or hb.numel() < words:
            hb = self.host[which] = torch.empty(words + 1024, dtype=torch.int32, pin_memory=True)
        with torch.cuda.stream(self.side):
            hb[:words].copy_(self.bufs[which][:words], non_blocking=True)
        hev = torch.cuda.Event()
        hev.record(self.side)
        self.cur, self.key, self.words, self.ready, self.host_ready = which, (mt.tobytes(), pos), words, ev, hev

    def acquire(self, mt, pos, words):
        """Buffer holding >= words outputs from (mt,pos); the current stream is made to wait for it."""
        self.flush()
        with self.lock:
            if self.key != (mt.tobytes(), pos) or self.words < words:
                self._generate(self.cur ^ 1, mt, pos, words)
            _cur_stream().wait_event(self.ready)
            return self.bufs[self.cur]

    def acquire_nowait(self, mt, pos, words):
        """As acquire, but the caller orders its consumer behind `self.ready` itself (mscs_forward_chain makes the
        sampling stream wait for it)."""
        self.flush()
        with self.lock:
            if self.key != (mt.tobytes(), pos) or self.words < words:
                self._generate(self.cur ^ 1, mt, pos, words)
            return self.bufs[self.cur]

    def state_after(self, mt, pos, total):
        """Generator state (mt', pos') after `total` draws from (mt, pos).  The stream buffer holds the RAW state
        words, so the new state array is simply the 624-word block the next draw falls into: it is read back
        (2.5 KB on a private stream) instead of recomputing ~800 block regenerations on the host (~100 us at cfg-2).
        Same convention as mscs_mt19937_advance_host: pos in 1..624, an exhausted block is not regenerated."""
        if total <= 0:
            return mt, pos
        blk = (pos + total - 1) // _MT_N
        newpos = pos + total - blk * _MT_N
        if blk == 0:
            return mt, newpos
        off = blk * _MT_N - pos
        with self.lock:
            buf = self.bufs[self.cur]
            if self.key != (mt.tobytes(), pos) or off + _MT_N > self.words:
                return None
            if self.host_ready is not None and self.host[self.cur] is not None:
                self.host_ready.synchronize()       # complete long ago (the mirror follows the generator kernel)
                host = self.host[self.cur][off:off + _MT_N].numpy().view(np.uint32).copy()
            else:
                host = np.empty(_MT_N, dtype=np.uint32)
                _lib.check(_lib.load().mscs_read_to_host(host.ctypes.data, buf.data_ptr() + 4 * off, 4 * _MT_N,
                                                         C.c_void_p(self.ready.cuda_event),
                                                         C.c_void_p(self.copy.cuda_stream)), "mscs_read_to_host")
        return host, newpos

    def release_and_prefetch(self, mt_next, pos_next, words, defer=False):
        """defer: only note the request; `flush` launches it.  The forward of a training step defers: between the plan
        fetch and the launch of the backward the host races ~0.35 ms of queued GPU work (cfg-2), and the generator
        launch (state upload, kernel, events: ~40 us) can as well follow the backward's launches."""
        with self.lock:
            ev = torch.cuda.Event()
            ev.record(_cur_stream())
            self.last_use[self.cur] = ev
            if defer:
                self.pending = (mt_next, pos_next, words)
            else:
                self.pending = None
                self._generate(self.cur ^ 1, mt_next, pos_next, words)

    def flush(self):
        """Launches a deferred prefetch, if any (after the backward has been enqueued; the next acquire does it too)."""
        if self.pending is None:
            return
        with self.lock:
            p, self.pending = self.pending, None
            if p is not None:
                self._generate(self.cur ^ 1, *p)


_stream_caches = {}


def _stream_cache(dev):
    c = _stream_caches.get(dev)
    if c is None:
        c = _stream_caches[dev] = _StreamCache(dev)
    return c


# ---- K1 -----------------------------------------------------------------------------------
def sample_anchors(labels, feat_hw, spec, mt_state=None, defer_rng=False):
    """All scales of one call.  ``feat_hw``: [(h, w)] per scale.  ``mt_state``: None = consume the
    torch CPU default generator exactly as the reference does, or an explicit (uint32[624], pos)."""
    lib = _lib.load()
    _require_device(labels)
    if labels.dtype not in (torch.int64, torch.int16):
        labels = labels.long()
    labels = labels.contiguous()
    n, H, W = labels.shape
    S = len(feat_hw)
    cfg = _lib.SampleCfg()
    cfg.n, cfg.H, cfg.W, cfg.num_scales = n, H, W, S
    for s, (h, w) in enumerate(feat_hw):
        cfg.fh[s], cfg.fw[s] = h, w
    cfg.num_classes, cfg.min_views = spec.num_classes, spec.min_views
    cfg.max_views, cfg.max_total = spec.max_views, spec.max_total
    dev = labels.device
    ws_bytes = lib.mscs_sample_workspace_bytes(C.byref(cfg))
    if ws_bytes == 0:
        raise RuntimeError("mscs_sample_workspace_bytes: " + lib.mscs_last_error().decode())
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    plan_dev = torch.empty(S * C.sizeof(_lib.ScalePlan), dtype=torch.uint8, device=dev)
    st = _stream()
    fn, fname = _plan_entry(lib, labels)
    _lib.check(fn(C.byref(cfg), labels.data_ptr(), ws.data_ptr(), plan_dev.data_ptr(), st), fname)
    plan = (_lib.ScalePlan * S)()
    _lib.check(lib.mscs_plan_fetch(plan_dev.data_ptr(), plan, S, st), "mscs_plan_fetch")
    for s in range(S):
        if plan[s].error == 1:   # reference: torch.min() of an empty tensor raises (V2.py:110)
            raise RuntimeError(f"scale {s}: no (image, class) pair has >= min_views_per_class="
                               f"{spec.min_views} pixels (the reference raises here too, V2.py:110)")
        if plan[s].error == 2:   # reference: 0-d squeeze then .shape[0] raises (V2.py:119-121)
            raise IndexError(f"scale {s}: a kept class has a single pixel (the reference raises here too)")
    total = sum(int(plan[s].draws) for s in range(S))
    own_rng = mt_state is None
    max_draws = int(lib.mscs_sample_max_draws(C.byref(cfg)))
    if own_rng:
        mt, pos = torch_mt_state()
        draws = _stream_cache(dev).acquire(mt, pos, max_draws)
    else:
        mt, pos = np.ascontiguousarray(mt_state[0], dtype=np.uint32), int(mt_state[1])
        draws = torch.empty(total + 64 + 1024, dtype=torch.int32, device=dev)
        _lib.check(lib.mscs_mt19937_stream(mt.ctypes.data_as(C.c_void_p), pos, C.c_uint64(total),
                                           draws.data_ptr(), st), "mscs_mt19937_stream")
    A = spec.num_classes
    # one int32 slab for every per-scale index array
    offs, off = [], 0
    for s in range(S):
        N, T = plan[s].N, plan[s].T
        cur = []
        for x in (N, 2 * T, N, N, A + 1):
            cur.append(off)
            off += (x + 15) // 16 * 16
        offs.append(cur)
    slab = torch.empty(off, dtype=torch.int32, device=dev)
    out = [ScaleSample(plan[s].T, plan[s].V, plan[s].N, bool(plan[s].log_flag), plan[s].dl_h, plan[s].dl_w,
                       slab, offs[s], A) for s in range(S)]
    arrs = [[out[s].ptr(k) for s in range(S)] for k in range(5)]
    _lib.check(lib.mscs_sample_select(C.byref(cfg), plan, ws.data_ptr(), draws.data_ptr(),
                                      *[_lib.ptr_array(a) for a in arrs], None, st), "mscs_sample_select")

    def finish_rng():
        """Publish the generator state the reference would leave behind and start producing the
        next call's stream.  Deferred by the caller until the tensor kernels are enqueued."""
        if own_rng:
            mt2, pos2 = torch_mt_advance(mt, pos, total)
            _stream_cache(dev).release_and_prefetch(mt2, pos2, max_draws)

    if defer_rng:
        return out, finish_rng
    finish_rng()
    return out


# ---- K2 -----------------------------------------------------------------------------------
@dataclass
class AnchorSet:
    N: int
    C: int
    C_pad: int
    bf16: torch.Tensor       # (N_pad, C_pad) bf16 unit rows (zero padded)
    f32: torch.Tensor        # (N, C) fp32 unit rows
    inv_norm: torch.Tensor   # (N,)


def gather_normalize(feat, sample):
    lib = _lib.load()
    n, Cc, h, w = feat.shape
    N = sample.N
    C_pad, N_pad = (Cc + 63) // 64 * 64, (N + 255) // 256 * 256
    dev = feat.device
    bf = torch.empty((N_pad, C_pad), dtype=torch.bfloat16, device=dev)
    f32 = torch.empty((N, Cc), dtype=torch.float32, device=dev)
    inv = torch.empty((N,), dtype=torch.float32, device=dev)
    _lib.check(lib.mscs_gather_normalize(feat.data_ptr(), n, Cc, h * w, sample.pix.data_ptr(), N, bf.data_ptr(),
                                         f32.data_ptr(), inv.data_ptr(), _stream()), "mscs_gather_normalize")
    return AnchorSet(N=N, C=Cc, C_pad=C_pad, bf16=bf, f32=f32, inv_norm=inv)


# ---- K3 / K4 ------------------------------------------------------------------------------
@dataclass
class SimState:
    job: _lib.SimJob
    keep: list                      # tensors the job points into
    term_loss: torch.Tensor
    total: torch.Tensor
    num_ms: int
    cs_logged: List[int]            # indices (into term_loss) of the cs terms that go to cs_losses


def build_job(spec, samples, sets, single_scale):
    """Terms of one call: one single-scale term per scale (V2.py:55 via _ms.py:53-59) and, when
    cross_scale_contrast, scale 0 against the deepest and second-deepest scales (_ms.py:62-80)."""
    S = len(sets)
    terms = [(s, s, True, spec.weights[s], spec.temperature, False) for s in range(S)]
    cs_logged = []
    if spec.cross_scale and not single_scale:
        assert S > 1, "cross_scale_contrast needs at least two scales (_ms.py:63-64)"
        need_dk = not spec.detach_deepest
        terms.append((0, S - 1, False, spec.w_high_low, spec.cs_temperature, need_dk))
        if not spec.detach_deepest:          # _ms.py:66-70: not logged when the deepest scale is detached
            cs_logged.append(len(terms) - 1)
        if S > 2:
            terms.append((0, S - 2, False, spec.w_high_mid, spec.cs_temperature, need_dk))
            cs_logged.append(len(terms) - 1)
    if len(terms) > _lib.MAX_TERMS:
        raise ValueError(f"{len(terms)} loss terms exceed the supported {_lib.MAX_TERMS}")
    dev = sets[0].bf16.device
    n_rows = [sets[a].N for a, *_ in terms]
    stats = torch.zeros(3 * sum(n_rows), dtype=torch.float32, device=dev)
    coefs = torch.empty(2 * sum(n_rows), dtype=torch.float32, device=dev)
    out = torch.empty(len(terms) + 2, dtype=torch.float32, device=dev)      # term losses, total, inf/NaN flag
    job = _lib.SimJob()
    job.num_terms, job.C_pad, job.num_classes = len(terms), sets[0].C_pad, spec.num_classes
    so = co = 0
    for i, (a, k, self_mask, weight, tau, need_dk) in enumerate(terms):
        t = job.terms[i]
        t.a_bf16, t.k_bf16 = sets[a].bf16.data_ptr(), sets[k].bf16.data_ptr()
        t.a_cls, t.k_seg = samples[a].cls.data_ptr(), samples[k].seg.data_ptr()
        t.k_cls, t.a_seg = samples[k].cls.data_ptr(), samples[a].seg.data_ptr()
        t.N1, t.N2, t.self_mask, t.need_dk = sets[a].N, sets[k].N, int(self_mask), int(need_dk)
        t.temperature, t.weight, t.a_set, t.k_set = tau, weight, a, k
        n1 = sets[a].N
        t.neg_sum = stats[so:so + n1].data_ptr()
        t.pos_sum = stats[so + n1:so + 2 * n1].data_ptr()
        t.s_sum = stats[so + 2 * n1:so + 3 * n1].data_ptr()
        t.coef_s = coefs[co:co + n1].data_ptr()
        t.coef_pn = coefs[co + n1:co + 2 * n1].data_ptr()
        so += 3 * n1
        co += 2 * n1
    job.term_loss, job.total_loss = out.data_ptr(), out[len(terms):].data_ptr()
    total = torch.empty((), dtype=torch.float32, device=dev)
    job.total_out = total.data_ptr()
    work = torch.empty(_lib.load().mscs_sim_workspace_bytes(C.byref(job)), dtype=torch.uint8, device=dev)
    job.work = work.data_ptr()
    return SimState(job=job, keep=[stats, coefs, out, work], term_loss=out[:len(terms)], total=total,
                    num_ms=S, cs_logged=cs_logged)


def sim_forward(state):
    _lib.check(_lib.load().mscs_sim_forward(C.byref(state.job), _stream()), "mscs_sim_forward")


def sim_backward(state, sets, grad_out):
    lib = _lib.load()
    dev = sets[0].bf16.device
    dFs = [torch.zeros((a.N, a.C_pad), dtype=torch.float32, device=dev) for a in sets]
    ptrs = [0] * _lib.MAX_SCALES
    lds = (C.c_int32 * _lib.MAX_SCALES)()
    for s, d in enumerate(dFs):
        ptrs[s], lds[s] = d.data_ptr(), d.shape[1]
    g = grad_out.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
    with _timed("sim_bwd"):
        _lib.check(lib.mscs_sim_backward(C.byref(state.job), g.data_ptr(), _lib.ptr_array(ptrs), lds, _stream()),
                   "mscs_sim_backward")
    return dFs


class _GradBuffers:
    """Dense feature gradients zero-filled ahead of time on a side stream (the zero fill is the
    largest HBM term of the whole path, SURVEY.md §8d, and does not depend on any result).  One slab for all
    scales and one fill: the per-scale tensors handed to autograd are views of it, in the dtype of the maps."""
    _side = {}

    def __init__(self, feats, needs, nhwc=False, extra=0):
        dev = feats[0].device
        side = self._side.get(dev)
        if side is None:
            side = self._side[dev] = torch.cuda.Stream(device=dev)
        # bytes per buffer, each rounded up to 16 (row stores of the scatter; mixed dtypes stay aligned)
        sizes = [(f.numel() * f.element_size() + 15) // 16 * 16
                 if (need and (nhwc or (f.shape[2] * f.shape[3]) % 8 == 0)) else 0 for f, need in zip(feats, needs)]
        # `extra` floats after the dense gradients: the gradient-row slab (dF) of the backward, zeroed by the same fill
        dense = (sum(sizes) + 255) // 256 * 256       # dF starts 256-byte aligned (vector reductions / loads)
        self.slab = torch.empty(dense + 4 * extra if extra else sum(sizes), dtype=torch.uint8, device=dev)
        self.dF = self.slab[dense:].view(torch.float32) if extra else None
        self.bufs, off = [], 0
        for f, n_ in zip(feats, sizes):
            if not n_:
                self.bufs.append(None)
            elif nhwc:      # same (n, C, h, w) shape, channels-last strides like the input
                n, Cc, h, w = f.shape
                buf = self.slab[off:off + f.numel() * f.element_size()].view(f.dtype)
                self.bufs.append(buf.view(n, h, w, Cc).permute(0, 3, 1, 2))
            else:
                self.bufs.append(self.slab[off:off + f.numel() * f.element_size()].view(f.dtype).view(f.shape))
            off += n_
        self.side, self.ready = side, None

    def start_fill(self, extra=None):
        """Zero-fill on the side stream, ordered after what the main stream has enqueued so far.  `extra`: one more
        (address, bytes) region cleared by the same call (pooled mode: the gradient rows in the exchange slab)."""
        side = self.side
        side.wait_stream(_cur_stream())
        if self.slab.numel() or extra:
            regions = ([(self.slab.data_ptr(), self.slab.numel())] if self.slab.numel() else []) + \
                ([extra] if extra else [])
            ptrs = _lib.ptr_array([r[0] for r in regions])
            if TIMING is not None:      # bench.py: the fill's own duration, on the stream it runs on
                e0 = torch.cuda.Event(enable_timing=True)
                e0.record(side)
            _lib.check(_lib.load().mscs_fill_bytes(ptrs, (C.c_int32 * len(regions))(*([0] * len(regions))),
                                                   (C.c_size_t * len(regions))(*[r[1] for r in regions]), len(regions),
                                                   C.c_void_p(side.cuda_stream)), "mscs_fill_bytes")
            if TIMING is not None:
                e1 = torch.cuda.Event(enable_timing=True)
                e1.record(side)
                TIMING.setdefault("zero_fill", []).append((e0, e1))
            if self.slab.numel():
                self.slab.record_stream(side)
        self.ready = torch.cuda.Event()
        self.ready.record(side)

    def take(self, s):
        """The pre-zeroed buffer of scale s (once: a second backward falls back to zero-fill)."""
        b, self.bufs[s] = self.bufs[s], None
        return b

    def take_dF(self):
        """The pre-zeroed gradient-row slab (once)."""
        d, self.dF = self.dF, None
        return d


# ---- pooled cross-batch mode: exchange over NVLink peer memory ---------------------------------
class _SymSlab:
    """One rank's view of the exchange slabs of all ranks (csrc/xchg.cu): `local` = address of the own slab, `peers` =
    ctypes array of every rank's slab as mapped here (peers[rank] == local), `epoch` = barrier counter (identical
    sequence on every rank), `parity` = which half the next step uses."""

    def __init__(self, local, peer_ptrs, keep=None):
        self.local, self.peers, self.keep = local, _lib.ptr_array(peer_ptrs), keep
        self.epoch, self.parity = 0, 0


class TorchDistComm:
    """Pooled mode over the GPUs of one box, one process per GPU.  torch.distributed (NCCL) carries only the two
    tiny control-plane exchanges (class histograms, IPC handles); the data plane -- normalised key rows, row
    statistics, gradient rows -- is written / read by the library's own kernels over NVLink peer memory, ordered by a
    device-side flag barrier (mscs_xchg_*)."""

    def __init__(self, group=None, barrier_timeout_s=20.0):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.owns_rng = True
        self.timeout = barrier_timeout_s
        if self.world > _lib.MAX_RANKS:
            raise ValueError(f"pooled mode supports up to {_lib.MAX_RANKS} ranks (one box), got {self.world}")

    def all_gather(self, t):
        out = torch.empty(self.world * t.numel(), dtype=t.dtype, device=t.device)
        self.dist.all_gather_into_tensor(out, t.reshape(-1), group=self.group)
        return out

    def symmetric(self, nbytes, dev):
        """Collective: every rank allocates its exchange slab (cudaMalloc, zeroed) and maps everybody else's."""
        lib = _lib.load()
        ptr, handle = C.c_void_p(), C.create_string_buffer(_lib.IPC_HANDLE_BYTES)
        _lib.check(lib.mscs_xchg_alloc(nbytes, C.byref(ptr), handle), "mscs_xchg_alloc")
        mine = torch.tensor(list(handle.raw), dtype=torch.uint8, device=dev)
        handles = self.all_gather(mine).cpu().numpy().reshape(self.world, _lib.IPC_HANDLE_BYTES)
        peers = []
        for r in range(self.world):
            if r == self.rank:
                peers.append(ptr.value)
                continue
            q = C.c_void_p()
            _lib.check(lib.mscs_xchg_open(handles[r].tobytes(), C.byref(q)), "mscs_xchg_open")
            peers.append(q.value)
        return _SymSlab(ptr.value, peers)

    def barrier(self, slab):
        """Device-side barrier on the current stream (no host wait)."""
        slab.epoch += 1
        _lib.check(_lib.load().mscs_xchg_barrier(slab.peers, self.world, self.rank, slab.epoch, self.timeout, _stream()),
                   "mscs_xchg_barrier")


class ThreadComm:
    """In-process emulation of `world` ranks on ONE device (one Python thread per rank): the slabs of all "ranks" live
    in one address space (the peer stores of the kernels are plain local stores) and the barrier is a host barrier
    around a device synchronisation.  Test infrastructure for the pooled mode's host logic and row-range kernels."""

    class _Shared:
        def __init__(self, world):
            import threading
            self.world, self.slots, self.result = world, [None] * world, None
            self.barrier = threading.Barrier(world)

    def __init__(self, shared, rank):
        self.sh, self.rank, self.world = shared, rank, shared.world
        self.owns_rng = rank == 0          # the CPU generator is process-global: one rank publishes it

    def _exchange(self, t, combine):
        sh = self.sh
        sh.slots[self.rank] = t
        sh.barrier.wait()
        if self.rank == 0:
            torch.cuda.synchronize()
            sh.result = combine(sh.slots)
            torch.cuda.synchronize()
        sh.barrier.wait()
        res = sh.result
        sh.barrier.wait()
        return res

    def all_gather(self, t):
        return self._exchange(t, lambda ts: torch.cat([x.reshape(-1) for x in ts])).clone()

    def symmetric(self, nbytes, dev):
        mine = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        ptrs = self._exchange(mine.data_ptr(), lambda xs: list(xs))
        return _SymSlab(mine.data_ptr(), list(ptrs), keep=mine)

    def barrier(self, slab):
        slab.epoch += 1
        torch.cuda.synchronize()
        self.sh.barrier.wait()


def shard_rows(N, world, rank):
    """128-aligned row range of `rank` among `world` ranks over N sorted anchor rows."""
    per = ((N + 127) // 128 + world - 1) // world * 128
    b = min(N, rank * per)
    e = min(N, b + per)
    return b, e


# ---- fused host path of the autograd Function -------------------------------------------------
class _StepPlan:
    """Everything of a call that depends only on shapes and configuration, computed once and cached:
    C structs, buffer layouts sized by upper bounds (N <= max_features_total), the term list.  With it
    every allocation and the MT19937 stream lookup happen BEFORE the one host sync of the forward
    pass, and only three kinds of C calls remain after it (select, gather, similarity forward)."""

    def __init__(self, dev, label_shape, feat_shapes, spec, single_scale, world=1, rank=0, nhwc=False):
        lib = _lib.load()
        self.dev, self.spec, self.single_scale = dev, spec, single_scale
        self.nhwc = nhwc            # feature maps are channels-last in memory ([n][h][w][C]): row gather / scatter
        self.world, self.rank = world, rank
        n, H, W = label_shape
        self.n_local, self.n_global = n, n * world
        self.S = S = len(feat_shapes)
        self.A = A = spec.num_classes
        self.feat_shapes = feat_shapes
        cfg = self.cfg = _lib.SampleCfg()
        cfg.n, cfg.H, cfg.W, cfg.num_scales = n, H, W, S
        for s, shp in enumerate(feat_shapes):
            cfg.fh[s], cfg.fw[s] = shp[2], shp[3]
        cfg.num_classes, cfg.min_views = A, spec.min_views
        cfg.max_views, cfg.max_total = spec.max_views, spec.max_total
        if world > 1:
            cfg.n_global, cfg.image_base = n * world, n * rank
        self.ws_bytes = lib.mscs_sample_workspace_bytes(C.byref(cfg))
        if self.ws_bytes == 0:
            raise RuntimeError("mscs_sample_workspace_bytes: " + lib.mscs_last_error().decode())
        self.max_draws = int(lib.mscs_sample_max_draws(C.byref(cfg)))
        # upper bound of views per pair (V2.py:64-84): V <= max_views_per_class unless that is 1, and V*T <= max_total
        self.v_cap = min(spec.max_total, 16384) if spec.max_views == 1 else min(spec.max_views, spec.max_total, 16384)
        self.C = Cc = feat_shapes[0][1]
        for shp in feat_shapes:
            if shp[1] != Cc:
                raise ValueError("all feature maps must have the same number of channels")
        self.C_pad = (Cc + 63) // 64 * 64
        Tcap = n * world * (A - 1)
        self.Ncap = [min(spec.max_total, n * world * shp[2] * shp[3]) for shp in feat_shapes]
        self.counts_off = [int(lib.mscs_sample_counts_offset(C.byref(cfg), s)) for s in range(S)]
        al = lambda x, a=16: (x + a - 1) // a * a
        # int32 slab: idx_ref, pair_ref, pix, cls, seg per scale
        self.ioff, off = [[0] * 5 for _ in range(S)], 0
        for k in (0, 1, 2, 4, 3):           # the class arrays (k = 3) last and adjacent: one all-reduce in pooled mode
            if k == 3:
                self.cls_begin = off
            for s in range(S):
                self.ioff[s][k] = off
                off += al((self.Ncap[s], 2 * Tcap, self.Ncap[s], self.Ncap[s], A + 1)[k])
        self.islab_n = off
        # fp32 slab: unit rows + inverse norms per scale;  bf16 slab: padded operand matrices
        self.foff, off = [], 0
        for s in range(S):
            self.foff.append((off, off + al(self.Ncap[s] * Cc)))
            off += al(self.Ncap[s] * Cc) + al(self.Ncap[s])
        self.fslab_n = off
        self.boff, off = [], 0
        for s in range(S):
            self.boff.append(off)
            off += al(self.Ncap[s], 256) * self.C_pad
        self.bslab_n = off
        # terms (V2.py:55 via _ms.py:53-59; cross-scale _ms.py:62-80)
        terms = [(s, s, True, spec.weights[s], spec.temperature, False) for s in range(S)]
        self.cs_logged = []
        if spec.cross_scale and not single_scale:
            assert S > 1, "cross_scale_contrast needs at least two scales (_ms.py:63-64)"
            need_dk = not spec.detach_deepest
            terms.append((0, S - 1, False, spec.w_high_low, spec.cs_temperature, need_dk))
            if not spec.detach_deepest:
                self.cs_logged.append(len(terms) - 1)
            if S > 2:
                terms.append((0, S - 2, False, spec.w_high_mid, spec.cs_temperature, need_dk))
                self.cs_logged.append(len(terms) - 1)
        if len(terms) > _lib.MAX_TERMS:
            raise ValueError(f"{len(terms)} loss terms exceed the supported {_lib.MAX_TERMS}")
        self.terms = terms
        self.soff, off = [], 0          # stats: neg, pos, S per term (zero-initialised)
        for a, *_ in terms:
            self.soff.append(off)
            off += 3 * al(self.Ncap[a])
        self.stats_n = off
        self.coff, off = [], 0          # coefficients + per-term losses + total
        for a, *_ in terms:
            self.coff.append(off)
            off += 2 * al(self.Ncap[a])
        self.out_off = off
        self.misc_n = off + al(len(terms) + 2)      # term losses, total, inf/NaN flag
        job = _lib.SimJob()
        job.num_terms, job.C_pad, job.num_classes = len(terms), self.C_pad, A
        for i, (a, k, self_mask, weight, tau, need_dk) in enumerate(terms):
            t = job.terms[i]
            t.N1, t.N2 = self.Ncap[a], self.Ncap[k]
            t.self_mask, t.need_dk, t.temperature, t.weight, t.a_set, t.k_set = int(self_mask), int(need_dk), tau, \
                weight, a, k
        self.work_bytes = lib.mscs_sim_workspace_bytes(C.byref(job))
        self.dF_off, off = [], 0
        for s in range(S):
            self.dF_off.append(off)
            off += (self.Ncap[s] + 128 * world) * self.C_pad      # slack: `world` 128-aligned row blocks (pooled mode)
        self.dF_n = off
        # single-process calls: ONE allocation per forward; byte offsets (256-aligned) of its parts
        self.slot_sizes = [shp[0] * shp[2] * shp[3] if (shp[2] * shp[3]) % 8 == 0 else 0 for shp in feat_shapes]
        parts = [("ws", self.ws_bytes), ("plan", S * C.sizeof(_lib.ScalePlan)), ("work", self.work_bytes),
                 ("stats", 4 * self.stats_n), ("misc", 4 * self.misc_n), ("fslab", 4 * self.fslab_n),
                 ("islab", 4 * self.islab_n), ("slot", 4 * sum(self.slot_sizes)), ("bslab", 2 * self.bslab_n),
                 ("dF", 4 * self.dF_n)]
        self.slab_off, off = {}, 0
        for name, nbytes in parts:
            self.slab_off[name] = off
            off += (nbytes + 255) // 256 * 256
        self.slab_bytes = off
        self.ws_pool = []           # reusable _Workspace objects of the single-process fast path
        # pooled mode: layout of the exchange slab (identical on every rank): barrier flags, then per step parity the
        # operand matrices (bf16), the row statistics and the gradient rows.  Two parities: a rank that runs ahead
        # writes the next step's rows while a slower rank still reads this step's (DESIGN.md section 6).
        self.x_off, off = [], 256
        for _par in range(2):
            d = {}
            for name, nbytes in (("b", 2 * self.bslab_n), ("stats", 4 * self.stats_n), ("dF", 4 * self.dF_n)):
                d[name] = off
                off += (nbytes + 255) // 256 * 256
            self.x_off.append(d)
        self.x_bytes = off
        self.xslab = None            # _SymSlab, created by the first pooled call (collective)


_step_plans = {}


def _step_plan(dev, label_shape, feat_shapes, spec, single_scale, world=1, rank=0, nhwc=False, create=True):
    """The cached plan of these shapes and this configuration (create=False: None when no call has made it yet)."""
    key = (dev, tuple(label_shape), tuple(feat_shapes), spec.num_classes, spec.temperature, spec.cs_temperature,
           spec.min_views, spec.max_views, spec.max_total, tuple(spec.weights), spec.cross_scale,
           spec.detach_deepest, spec.w_high_low, spec.w_high_mid, single_scale, world, rank, nhwc)
    p = _step_plans.get(key)
    if p is None and create:
        p = _step_plans[key] = _StepPlan(dev, label_shape, feat_shapes, spec, single_scale, world, rank, nhwc)
    return p


def fast_path_ok(spec, world):
    """Single process and selection shared memory within limits: the device-driven order can be used."""
    v_cap = min(spec.max_total, 16384) if spec.max_views == 1 else min(spec.max_views, spec.max_total, 16384)
    return world == 1 and v_cap * 12 <= 200 * 1024


def half_io_ok(sp, world):
    """Whether bf16 / fp16 feature maps are handed to the kernels as they are (no fp32 copy; the dense gradients are
    written in the maps' dtype): the single-process fast path with the channels-last row gather, or with the NCHW octet
    gather and the one-pass dense writer.  Every other route -- pooled mode, planes that are not a multiple of 8
    pixels -- converts the maps to fp32 first and the gradients back afterwards."""
    if not fast_path_ok(sp.spec, world):
        return False
    return sp.nhwc or all(sp.slot_sizes)


def channels_last_ok(spec, world, feats):
    """Channels-last feature maps (memory order [n][h][w][C]) are consumed as they are by the single-process fast path:
    an anchor is then one contiguous row (gather / scatter become row copies)."""
    return fast_path_ok(spec, world) and all(
        f.dim() == 4 and f.is_contiguous(memory_format=torch.channels_last) and not f.is_contiguous() for f in feats)


# first call index of graph replays: eager calls count up from 0 and never get here
GRAPH_CALL_BASE = 2 ** 62


def graph_mode(spec, world, single_scale, labels, feats, counter, plan_of=None):
    """Whether this call is being captured into a CUDA graph (``torch.cuda.graph``), which the single-process fast path
    with sampler='philox' supports: the call then enqueues work without ever waiting for the host (the row counts stay
    on the device, the Philox call index is read from ``counter``).  Everything that cannot be captured raises a
    RuntimeError here, before anything is enqueued, so that the capture still ends cleanly.  Outside a capture: False
    (the eager path, unchanged).  ``plan_of(nhwc)``: the caller's cached plan of these inputs, or None before its first
    eager call (default: the step plan of the loss classes)."""
    if not (feats[0].is_cuda and torch.cuda.is_current_stream_capturing()):      # (a CUDA tensor: a runtime exists)
        return False

    def refuse(why):
        raise RuntimeError(f"the contrastive loss cannot be captured in a CUDA graph: {why}")

    if world > 1:
        refuse("the pooled mode (comm) exchanges control data through the host")
    if spec.sampler != "philox":
        refuse("sampler='reference' advances the torch CPU generator by a label-dependent number of draws; "
               "use sampler='philox'")
    if single_scale and spec.cross_scale:
        refuse("DenseContrastiveLossV2 with cross_scale_contrast=True returns sampled features of a data-dependent shape")
    if not fast_path_ok(spec, world):
        refuse("the selection table of this configuration exceeds the device-driven path's shared memory")
    if any(f.device != feats[0].device for f in feats) or labels.device != feats[0].device:
        refuse("labels and feature maps must already be on the GPU")
    nhwc = channels_last_ok(spec, world, feats)
    if not nhwc and any((f.shape[2] * f.shape[3]) % 8 for f in feats):
        refuse("feature planes that are not a multiple of 8 pixels take the host-driven path")
    if plan_of is None:
        sp = _step_plan(feats[0].device, labels.shape, [tuple(f.shape) for f in feats], spec, single_scale, world, 0,
                        nhwc, create=False)
    else:
        sp = plan_of(nhwc)
    if sp is None or counter is None or counter.device != feats[0].device:
        refuse("run one eager call with the same shapes and configuration before capturing (warm-up)")
    return True


def _dense_grad_slab(shapes, dtypes, dev):
    """ONE allocation for the dense gradients of the one-pass writer: the slab, the per-scale gradient views (dtype
    `dtypes[j]`) and their byte offsets.  Planes are a multiple of 8 pixels, so every view starts 16-byte aligned (the
    writer's 16-byte stores)."""
    nbytes = [shp[0] * shp[1] * shp[2] * shp[3] * dt.itemsize for shp, dt in zip(shapes, dtypes)]
    slab = torch.empty(sum(nbytes), dtype=torch.uint8, device=dev)
    views, offs, off = [], [], 0
    for shp, dt, nb in zip(shapes, dtypes, nbytes):
        views.append(slab[off:off + nb].view(dt).view(shp))
        offs.append(off)
        off += nb
    return slab, views, offs


_hp_streams = {}


def _hp_stream(dev):
    """High-priority stream for the small, latency-bound sampling kernels: the 535 MB zero fill of the dense
    gradients runs concurrently on a default-priority side stream, and with equal priorities its ~100k blocks
    queue in front of them (+65 us on the sampling stage at cfg-2)."""
    st = _hp_streams.get(dev)
    if st is None:
        st = _hp_streams[dev] = torch.cuda.Stream(device=dev, priority=-1)
    return st


class _Ptr:
    """Address inside a slab (quacks like a tensor for data_ptr()): a torch view costs a few microseconds of
    Python each and most buffers of a step are only ever passed to the library as raw pointers."""
    __slots__ = ("p",)

    def __init__(self, p):
        self.p = p

    def data_ptr(self):
        return self.p


def _raise_plan_errors(plan, S, spec):
    for s in range(S):
        if plan[s].error == 1:   # reference: torch.min() of an empty tensor raises (V2.py:110)
            raise RuntimeError(f"scale {s}: no (image, class) pair has >= min_views_per_class="
                               f"{spec.min_views} pixels (the reference raises here too, V2.py:110)")
        if plan[s].error == 2:   # reference: 0-d squeeze then .shape[0] raises (V2.py:119-121)
            raise IndexError(f"scale {s}: a kept class has a single pixel (the reference raises here too)")
        if plan[s].error == 3:
            raise ValueError(f"scale {s}: {plan[s].V} views per class exceed the supported 16384")


def fetch_graph_plan(state):
    """Logged scalars [term losses..., total, inf/NaN flag] and plan records of the latest replay of a captured call, in
    ONE device->host copy (the only synchronisation).  Valid until the next replay of the graph."""
    sp, e = state.sp, state.entry
    nb = C.sizeof(_lib.ScalePlan) * sp.S
    off = sp.slab_off["plan"]
    raw = torch.cat([state.scalars.view(torch.uint8), e.slab[off:off + nb]]).cpu().numpy()
    ns = 4 * state.scalars.numel()
    plan = (_lib.ScalePlan * sp.S).from_buffer_copy(raw[ns:].tobytes())
    return raw[:ns].view(np.float32).tolist(), plan


def graph_samples(state, plan):
    """The ScaleSample list of a captured call's latest replay (views of the graph's workspace: the next replay
    overwrites them)."""
    sp, e = state.sp, state.entry
    return [ScaleSample(plan[s].T, plan[s].V, plan[s].N, bool(plan[s].log_flag), plan[s].dl_h, plan[s].dl_w, e.islab,
                        sp.ioff[s], sp.A) for s in range(sp.S)]


def _fill_job(job, sp, A, bbase, ibase, sbase, cbase, work_ptr):
    """Everything of the similarity job that follows from the slab layouts (sized by upper bounds)."""
    job.num_terms, job.C_pad, job.num_classes = len(sp.terms), sp.C_pad, A
    for i, (a, k, self_mask, weight, tau, need_dk) in enumerate(sp.terms):
        t = job.terms[i]
        t.a_bf16, t.k_bf16 = bbase + 2 * sp.boff[a], bbase + 2 * sp.boff[k]
        t.a_cls, t.k_seg = ibase + 4 * sp.ioff[a][3], ibase + 4 * sp.ioff[k][4]
        t.k_cls, t.a_seg = ibase + 4 * sp.ioff[k][3], ibase + 4 * sp.ioff[a][4]
        t.self_mask, t.need_dk = int(self_mask), int(need_dk)
        t.temperature, t.weight, t.a_set, t.k_set = tau, weight, a, k
        n1 = (sp.Ncap[a] + 15) // 16 * 16
        t.neg_sum = sbase + 4 * sp.soff[i]
        t.pos_sum = sbase + 4 * (sp.soff[i] + n1)
        t.s_sum = sbase + 4 * (sp.soff[i] + 2 * n1)
        t.coef_s = cbase + 4 * sp.coff[i]
        t.coef_pn = cbase + 4 * (sp.coff[i] + n1)
    job.work = work_ptr


class _Workspace:
    """Reusable device workspace of the single-process fast path, with every ctypes structure that depends only on
    its addresses built ONCE: the two similarity jobs (forward: upper bounds + device-resident row counts; backward:
    actual counts), the index-array pointer tables, the gather items, the byte-fill lists.  A call takes one from the
    pool of its step plan and the call's state gives it back when it dies (after the backward, or when the module
    replaces ``last_state``), so steady-state training ping-pongs between two of them and does no per-call slab
    allocation or structure filling.  The scalars handed to the caller live in a fresh tensor per call."""

    def __init__(self, sp, graph=False):
        dev, S, A = sp.dev, sp.S, sp.A
        # graph: allocated inside a CUDA graph capture and used by its replays only -- never returned to the pool
        self.graph = graph
        self.slab = slab = torch.empty(sp.slab_bytes, dtype=torch.uint8, device=dev)
        sb, so = slab.data_ptr(), sp.slab_off
        self.islab = slab[so["islab"]:so["islab"] + 4 * sp.islab_n].view(torch.int32)
        self.stats = slab[so["stats"]:so["stats"] + 4 * sp.stats_n].view(torch.float32)
        self.ws, self.plan_dev = sb + so["ws"], sb + so["plan"]
        self.fbase, self.bbase = sb + so["fslab"], sb + so["bslab"]
        self.fslab = _Ptr(self.fbase)
        self.slots, off = [], sb + so["slot"]
        for x in sp.slot_sizes:
            self.slots.append(_Ptr(off) if x else None)
            off += 4 * x
        ibase = self.islab.data_ptr()
        self.arrs = [_lib.ptr_array([ibase + 4 * sp.ioff[s][k] for s in range(S)]) for k in range(5)]
        if sp.nhwc:                 # row gather / scatter: no slot maps
            self.slots = [None] * S
        self.sarr = _lib.ptr_array([x.data_ptr() if x is not None else 0 for x in self.slots])
        # byte fills in front of the sampling chain: row statistics (0), slot maps (-1)
        self.dF_ptr = sb + so["dF"]          # gradient-row accumulators of the backward (cleared by the forward chain)
        self.fill_ptrs = _lib.ptr_array([sb + so["stats"], sb + so["slot"]])
        self.fill_vals = (C.c_int32 * 2)(0, 0xFF)
        self.fill_bytes = (C.c_size_t * 2)(4 * sp.stats_n, 0 if sp.nhwc else 4 * sum(sp.slot_sizes))
        # the backward's argument structures (one C call, csrc/step.cu): everything but the dense-gradient addresses
        self.bw_ptrs = _lib.ptr_array([self.dF_ptr + 4 * sp.dF_off[s] for s in range(S)] + [0] * (_lib.MAX_SCALES - S))
        self.bw_lds = (C.c_int32 * _lib.MAX_SCALES)(*([sp.C_pad] * S + [0] * (_lib.MAX_SCALES - S)))
        self.bw_items = (_lib.ScatterItem * S)()
        self.bw_rows = (C.c_int32 * S)()
        plan_sz = C.sizeof(_lib.ScalePlan)
        self.job_fwd, self.job_bwd = _lib.SimJob(), _lib.SimJob()
        for job in (self.job_fwd, self.job_bwd):
            _fill_job(job, sp, A, self.bbase, ibase, sb + so["stats"], sb + so["misc"], sb + so["work"])
        for i, (a, k, *_rest) in enumerate(sp.terms):
            t = self.job_fwd.terms[i]
            t.N1, t.N2 = sp.Ncap[a], sp.Ncap[k]
            t.n1_dev, t.n2_dev = self.plan_dev + a * plan_sz + 8, self.plan_dev + k * plan_sz + 8
        if sp.nhwc:
            self.gitems = (_lib.RowsItem * S)()
        else:
            self.gitems = (_lib.GatherItem * S)()
        for s in range(S):
            n, Cc, h, w = sp.feat_shapes[s]
            it = self.gitems[s]
            if sp.nhwc:
                it.pix, it.rows, it.C = ibase + 4 * sp.ioff[s][2], sp.Ncap[s], Cc
            else:
                it.n, it.C, it.plane, it.slot = n, Cc, h * w, self.slots[s].data_ptr()
            it.n_rows_dev = self.plan_dev + s * plan_sz + 8
            it.anc_bf16, it.anc_f32 = self.bbase + 2 * sp.boff[s], self.fbase + 4 * sp.foff[s][0]
            it.inv_norm = self.fbase + 4 * sp.foff[s][1]
        if not sp.nhwc:
            for s in range(S):
                n, Cc, h, w = sp.feat_shapes[s]
                it = self.bw_items[s]
                it.dF, it.ldF = self.dF_ptr + 4 * sp.dF_off[s], sp.C_pad
                it.anc_f32, it.inv_norm = self.fbase + 4 * sp.foff[s][0], self.fbase + 4 * sp.foff[s][1]
                it.slot, it.n, it.C, it.plane = self.slots[s].data_ptr(), n, Cc, h * w
        self.rows_dev = [self.plan_dev + s * plan_sz + 8 for s in range(S)]      # &plan_dev[s].N
        if graph:       # the backward of a captured call never sees the plan: upper bounds + device-resident counts
            for i, (a, k, *_rest) in enumerate(sp.terms):
                t = self.job_bwd.terms[i]
                t.N1, t.N2 = sp.Ncap[a], sp.Ncap[k]
                t.n1_dev, t.n2_dev = self.rows_dev[a], self.rows_dev[k]
            for s in range(S):
                self.bw_rows[s] = sp.Ncap[s]
                self.bw_items[s].n_rows_dev = self.rows_dev[s]
        self.plan = (_lib.ScalePlan * S)()
        self.last_stream = None
        self.philox = None          # stream buffer of the opt-in counter-based sampler (allocated on first use)
        # the whole forward as ONE C call (csrc/step.cu): every field that depends only on addresses, filled once
        ch = self.chain = _lib.ForwardChainArgs()
        ch.cfg, ch.v_cap, ch.workspace, ch.plan_dev = C.addressof(sp.cfg), sp.v_cap, self.ws, self.plan_dev
        ch.idx_ref, ch.pair_ref, ch.pix, ch.cls, ch.seg = (C.addressof(a) for a in self.arrs)
        ch.slot = C.addressof(self.sarr)
        ch.fill_ptrs, ch.fill_values = C.addressof(self.fill_ptrs), C.addressof(self.fill_vals)
        ch.fill_bytes, ch.n_fill = C.addressof(self.fill_bytes), 2
        ch.main_zero_ptr = self.dF_ptr
        ch.gather_kind = 1 if sp.nhwc else 0
        ch.gather_items, ch.job = C.addressof(self.gitems), C.addressof(self.job_fwd)


class _StepState:
    """Buffers of one call (kept alive for the backward)."""
    entry = None
    io_dtypes = None        # dtypes of the maps the kernels read and of the gradients they write (None: all fp32)

    def __del__(self):
        e, self.entry = self.entry, None
        if e is not None and not e.graph:
            self.sp.ws_pool.append(e)


def run_forward(sp, labels, feats32, needs, comm=None, philox=None, graph=False):
    """philox: None (reference stream: torch CPU generator) or (seed, call index) of the opt-in counter-based stream.
    feats32: fp32 maps, or bf16 / fp16 ones where half_io_ok(sp, world) holds (fast path only).
    graph: the call is captured into a CUDA graph (see graph_mode); philox is then (seed, int64 device call index)."""
    pooled = comm is not None and comm.world > 1
    # device-driven order (selection, gather and similarity forward enqueued before the host sees the plan): single
    # process, every plane a multiple of 8 pixels (slot maps), selection shared memory within limits
    if fast_path_ok(sp.spec, 1 if not pooled else comm.world) and (sp.nhwc or all(x != 0 for x in sp.slot_sizes)):
        return _run_forward_fast(sp, labels, feats32, needs, philox, graph)
    assert all(f.dtype == torch.float32 for f in feats32), "half maps are converted by the caller off the fast path"
    assert not sp.nhwc, "channels-last inputs are converted by the caller unless the fast path applies"
    if philox is not None:
        raise NotImplementedError("sampler='philox' is implemented for the single-process path with feature planes "
                                  "that are a multiple of 8 pixels (or channels-last inputs)")
    if pooled:
        return _run_forward_pooled(sp, labels, feats32, needs, comm)
    return _run_forward_general(sp, labels, feats32, needs)


def _finish_rng(sp, dev, mt, pos, total, defer=False):
    """Host-side generator bookkeeping, off the GPU's critical path: publish the state the reference's randperm
    calls would leave and start producing the next call's stream (defer: the launch follows the backward's)."""
    nxt = _stream_cache(dev).state_after(mt, pos, total)
    if nxt is None:
        mt2, pos2 = torch_mt_advance(mt, pos, total)
    else:
        mt2, pos2 = nxt
        if total > 0:
            _publish_mt_state(mt2, pos2)
    _stream_cache(dev).release_and_prefetch(mt2, pos2, sp.max_draws + _MT_N, defer)


def _run_forward_fast(sp, labels, feats32, needs, philox=None, graph=False):
    """Single process.  Selection, gather AND the similarity forward are driven by the DEVICE plan records and enqueued
    before the host looks at the plan: the one host wait of the forward pass (needed to raise the reference's errors
    and to size the backward) overlaps ~0.5 ms of queued GPU work instead of draining the stream.

    graph (CUDA graph capture): no host wait at all.  A fresh workspace of the graph's own; the backward structures
    carry the upper bounds and the device-resident row counts; errors, sampling results and the logging flag stay in
    the device plan records (read by the caller after a replay: fetch_graph_plan)."""
    lib = _lib.load()
    dev, S, A, spec = sp.dev, sp.S, sp.A, sp.spec
    st, cur = _stream(), _cur_stream()
    import time
    _t = time.perf_counter() if HOST_SEG is not None else 0.0
    if graph:
        e = _Workspace(sp, graph=True)
    else:
        e = sp.ws_pool.pop() if sp.ws_pool else _Workspace(sp)
    if e.last_stream is not None and e.last_stream != cur:
        cur.wait_stream(e.last_stream)          # reuse on another stream: order after its previous user
    e.last_stream = cur
    nt = len(sp.terms)
    out = torch.empty(nt + 2, dtype=torch.float32, device=dev)      # term losses, total, inf/NaN flag
    # the 0-d loss handed to the caller: a tensor of its own (not a view of `out`) -- the reference's LossWrapper
    # multiplies it IN PLACE (`loss *= weight`, LossWrapper.py:90), which autograd forbids on a view created inside
    # a custom Function, and which must not change the logged (unweighted) scalars
    total_t = torch.empty((), dtype=torch.float32, device=dev)
    for job in (e.job_fwd, e.job_bwd):
        job.term_loss, job.total_loss = out.data_ptr(), out.data_ptr() + 4 * nt
        job.total_out = total_t.data_ptr()
    # the small, latency-bound sampling kernels run on a high-priority stream (see _hp_stream)
    hp = _hp_stream(dev) if _USE_HP_STREAM else None
    st_s = C.c_void_p(hp.cuda_stream) if hp is not None else st
    ch = e.chain
    # MT19937 output stream of this call (normally produced ahead of time during the previous step): looked up
    # first, so that nothing but kernels sits between the launches of the sampling chain
    if philox is None:
        mt, pos = torch_mt_state()
        ch.draws = _stream_cache(dev).acquire_nowait(mt, pos, sp.max_draws + _MT_N).data_ptr()
        ch.wait_event = _stream_cache(dev).ready.cuda_event
    else:       # counter-based stream of this call: one small kernel in front of the chain, no generator state
        if e.philox is None:
            e.philox = torch.empty((sp.max_draws + 3) // 4 * 4 + 4, dtype=torch.int32, device=dev)
        if hp is not None:
            hp.wait_stream(cur)
        ch.draws, ch.wait_event = e.philox.data_ptr(), None
        if graph:       # call index in device memory, incremented behind the generator: every replay draws anew
            _lib.check(lib.mscs_philox_stream_dev(int(philox[0]) & (2 ** 64 - 1), philox[1].data_ptr(), sp.max_draws,
                                                  ch.draws, st_s), "mscs_philox_stream_dev")
        else:
            _lib.check(lib.mscs_philox_stream(int(philox[0]) & (2 ** 64 - 1), int(philox[1]), sp.max_draws, ch.draws,
                                              st_s), "mscs_philox_stream")
    _t = _seg("fwd: rng state + stream acquire", _t)
    # channels-last dense gradients + gradient rows: pre-zeroed on a side stream, sampled rows written by the backward
    # (NCHW maps need no fill: the backward writes their dense gradients in one streaming pass, see gather.cu).
    # Started here, next to the small sampling kernels: the fill (535 MB at cfg-2) costs ~70 us of step time
    # WHEREVER it runs (measured next to the sampling kernels, under the forward, under the backward, and as a
    # device-to-device copy from a persistent zero buffer) -- memset and D2D copies run on the SMs.
    gradbufs = _GradBuffers(feats32, needs, sp.nhwc, sp.dF_n) if (any(needs) and sp.nhwc) else None
    if gradbufs is not None:
        if graph:       # filled on the caller's stream: a forward captured without its backward leaves no open fork
            gradbufs.side = cur
        gradbufs.start_fill()
    _t = _seg("fwd: grad buffers", _t)
    ch.labels, ch.labels_i16 = labels.data_ptr(), int(labels.dtype == torch.int16)
    for s in range(S):
        e.gitems[s].feat, e.gitems[s].dtype = feats32[s].data_ptr(), _DTYPE_CODE[feats32[s].dtype]
    # gradient-row accumulators of the backward: cleared by the chain on the caller's stream, next to the sampling
    # kernels, when the one-pass dense writer will be used (otherwise they come pre-zeroed with the dense gradients, or
    # no gradient is wanted at all)
    dF_in_ws = any(needs) and gradbufs is None
    ch.main_zero_bytes = 4 * sp.dF_n if dF_in_ws else 0
    # the dense gradients of the backward (written in one pass, no fill): allocated HERE, before the host waits for the
    # plan, with the addresses entered into the backward's prebuilt structures -- not in the window after the wait
    grad_slab = grad_outs = None
    if dF_in_ws and all(needs) and not sp.nhwc:
        grad_slab, grad_outs, offs = _dense_grad_slab([f.shape for f in feats32], [f.dtype for f in feats32], dev)
        sbase = grad_slab.data_ptr()
        for j in range(S):
            e.bw_items[j].dfeat, e.bw_items[j].dtype = sbase + offs[j], _DTYPE_CODE[feats32[j].dtype]
    evs = None
    if TIMING is not None and TIMING_ALL and not graph:      # stage accounting (bench.py): five events INSIDE the chain
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        for i, ev in enumerate(evs):
            ev.record()         # creates the CUDA event; the chain records it again at its stage boundary
            ch.stage_events[i] = ev.cuda_event
    else:
        for i in range(5):
            ch.stage_events[i] = None
    if HOST_WAIT is not None:
        _t0 = time.perf_counter()
    plan = e.plan
    # ONE call: fills, hist -> tile scan -> plan -> select on the sampling stream (programmatic dependent launches; the
    # plan records travel to the host on a private stream), gather + similarity forward on the caller's stream, all
    # driven by the DEVICE plan records, then the one host wait of the forward pass (plan records only)
    _lib.check(lib.mscs_forward_chain(C.byref(ch), st_s, st, None if graph else plan), "mscs_forward_chain")
    if HOST_WAIT is not None:
        HOST_WAIT.append(time.perf_counter() - _t0)
    if evs is not None:
        TIMING.setdefault("sample", []).append((evs[0], evs[1]))
        TIMING.setdefault("gather", []).append((evs[2], evs[3]))
        TIMING.setdefault("sim_fwd", []).append((evs[3], evs[4]))
    _t = time.perf_counter() if HOST_SEG is not None else 0.0
    state = _StepState()
    state.sp, state.entry = sp, e          # (from here on an exception returns the workspace to the pool)
    state.graph = graph
    if graph:           # nothing is known on the host: the backward structures hold the device-count form already
        samples = None
    else:
        _raise_plan_errors(plan, S, spec)
        total = sum(int(plan[s].draws) for s in range(S))
        samples = [ScaleSample(plan[s].T, plan[s].V, plan[s].N, bool(plan[s].log_flag), plan[s].dl_h, plan[s].dl_w,
                               e.islab, sp.ioff[s], A) for s in range(S)]
        for i, (a, k, *_rest) in enumerate(sp.terms):      # the backward is launched with the actual counts
            t = e.job_bwd.terms[i]
            t.N1, t.N2 = samples[a].N, samples[k].N
    _t = _seg("fwd: after wait", _t)
    if philox is None:
        _finish_rng(sp, dev, mt, pos, total, defer=any(needs))
    _t = _seg("fwd: rng advance + prefetch", _t)
    state.job, state.samples, state.gradbufs, state.slots = e.job_bwd, samples, gradbufs, e.slots
    state.keep, state.stats, state.fslab = out, e.stats, e.fslab
    state.term_loss, state.total, state.scalars = out[:nt], total_t, out
    state.num_ms, state.cs_logged, state.comm = S, sp.cs_logged, None
    state.dF_ws = e.dF_ptr if dF_in_ws else None
    state.grad_slab, state.grad_outs = grad_slab, grad_outs
    state.io_dtypes = [f.dtype for f in feats32]
    if not graph:
        for s in range(S):
            e.bw_rows[s] = samples[s].N
    return state


def _run_forward_general(sp, labels, feats32, needs):
    """Host-driven order on one stream: plan, fetch (host sync), select, gather, forward.  Single process, planes that
    are not a multiple of 8 pixels (no slot maps) or selection shared memory beyond the fast path's limit."""
    lib = _lib.load()
    dev, S, A, spec = sp.dev, sp.S, sp.A, sp.spec
    st = _stream()
    i32, f32, u8 = torch.int32, torch.float32, torch.uint8
    ws = torch.empty(sp.ws_bytes, dtype=u8, device=dev)
    plan_dev = torch.empty(S * C.sizeof(_lib.ScalePlan), dtype=u8, device=dev)
    with _timed("sample"):
        fn, fname = _plan_entry(lib, labels)
        _lib.check(fn(C.byref(sp.cfg), labels.data_ptr(), ws.data_ptr(), plan_dev.data_ptr(), st), fname)
        sizes = sp.slot_sizes
        islab = torch.empty(sp.islab_n, dtype=i32, device=dev)
        fslab = torch.empty(sp.fslab_n, dtype=f32, device=dev)
        bslab = torch.empty(sp.bslab_n, dtype=torch.bfloat16, device=dev)
        stats = torch.zeros(sp.stats_n, dtype=f32, device=dev)
        misc = torch.empty(sp.misc_n, dtype=f32, device=dev)
        work = torch.empty(sp.work_bytes, dtype=u8, device=dev)
        # pixel -> row maps (filled by the selection kernel): drive the address-ordered gather and the
        # sector scatter of the backward
        slot_slab = torch.full((sum(sizes),), -1, dtype=i32, device=dev) if sum(sizes) else None     # one fill
        slots, off = [], 0
        for x in sizes:
            slots.append(slot_slab[off:off + x] if x else None)
            off += x
        gradbufs = _GradBuffers(feats32, needs, False, sp.dF_n) if any(needs) else None
        if gradbufs is not None:
            gradbufs.start_fill()
        mt, pos = torch_mt_state()
        draws = _stream_cache(dev).acquire(mt, pos, sp.max_draws + _MT_N)
        plan = (_lib.ScalePlan * S)()
        ibase = islab.data_ptr()
        arrs = [_lib.ptr_array([ibase + 4 * sp.ioff[s][k] for s in range(S)]) for k in range(5)]
        sarr = _lib.ptr_array([x.data_ptr() if x is not None else 0 for x in slots])
        fbase, bbase = fslab.data_ptr(), bslab.data_ptr()
        job = _lib.SimJob()
        _fill_job(job, sp, A, bbase, ibase, stats.data_ptr(), misc.data_ptr(), work.data_ptr())
        nt = len(sp.terms)
        mbase = misc.data_ptr()
        job.term_loss, job.total_loss = mbase + 4 * sp.out_off, mbase + 4 * (sp.out_off + nt)
        total_t = torch.empty((), dtype=f32, device=dev)      # own buffer, not a view (see _run_forward_fast)
        job.total_out = total_t.data_ptr()
        _lib.check(lib.mscs_plan_fetch(plan_dev.data_ptr(), plan, S, st), "mscs_plan_fetch")     # the host sync
        _raise_plan_errors(plan, S, spec)
        total = sum(int(plan[s].draws) for s in range(S))
        _lib.check(lib.mscs_sample_select(C.byref(sp.cfg), plan, ws.data_ptr(), draws.data_ptr(), *arrs, sarr, st),
                   "mscs_sample_select")
    samples = [ScaleSample(plan[s].T, plan[s].V, plan[s].N, bool(plan[s].log_flag), plan[s].dl_h, plan[s].dl_w,
                           islab, sp.ioff[s], A) for s in range(S)]
    with _timed("gather"):
        for s in range(S):
            n, Cc, h, w = sp.feat_shapes[s]
            if slots[s] is not None:
                _lib.check(lib.mscs_gather_normalize_sectors(feats32[s].data_ptr(), n, Cc, h * w, slots[s].data_ptr(),
                                                             samples[s].N, bbase + 2 * sp.boff[s],
                                                             fbase + 4 * sp.foff[s][0], fbase + 4 * sp.foff[s][1], st),
                           "mscs_gather_normalize_sectors")
            else:
                _lib.check(lib.mscs_gather_normalize(feats32[s].data_ptr(), n, Cc, h * w, samples[s].ptr(2),
                                                     samples[s].N, bbase + 2 * sp.boff[s], fbase + 4 * sp.foff[s][0],
                                                     fbase + 4 * sp.foff[s][1], st), "mscs_gather_normalize")
    for i, (a, k, *_rest) in enumerate(sp.terms):      # the plan-dependent fields of the job
        t = job.terms[i]
        t.N1, t.N2 = samples[a].N, samples[k].N
    with _timed("sim_fwd"):
        _lib.check(lib.mscs_sim_forward(C.byref(job), st), "mscs_sim_forward")
    _finish_rng(sp, dev, mt, pos, total)
    state = _StepState()
    state.sp, state.job, state.samples, state.gradbufs, state.slots = sp, job, samples, gradbufs, slots
    state.keep = (ws, islab, fslab, bslab, stats, misc, work, slot_slab)
    state.stats = stats
    state.fslab, state.term_loss = fslab, misc[sp.out_off:sp.out_off + nt]
    state.total = total_t
    state.scalars = misc[sp.out_off:sp.out_off + nt + 2]      # [term losses..., total, inf/NaN flag]: one copy for the logger
    state.num_ms, state.cs_logged, state.comm = S, sp.cs_logged, None
    return state


def _run_forward_pooled(sp, labels, feats32, needs, comm):
    """POOLED cross-batch mode (one process per GPU, each with its own images): the reference loss of the concatenated
    batch of all ranks.  Control plane over NCCL (class histograms: a few KB); data plane by the library's own kernels
    over NVLink peer memory (csrc/xchg.cu), ordered by three device-side barriers per step:

      K1 histograms -> all-gather of the (image, class) counts -> the SAME global plan on every rank -> selection of the
      local pixels (class ids of every row come from the plan: no exchange) -> K2 fused with the all-gather: each
      normalised bf16 row is stored into the same sorted row of EVERY rank's operand matrix -> barrier A ->
      K3 sweeps over this rank's anchor-row range against all keys -> its row statistics pushed to every peer ->
      barrier B -> finalise on all rows (every rank then holds the global loss and the coefficients of every row, so
      the backward needs no reduce-scatter) -> [backward: K4 over the rank's row range -> barrier C -> the scatter
      PULLS each gradient row of a local pixel from the rank that computed it]."""
    lib = _lib.load()
    dev, S, A, spec = sp.dev, sp.S, sp.A, sp.spec
    st = _stream()
    i32, f32, u8 = torch.int32, torch.float32, torch.uint8
    if not all(sp.slot_sizes):
        raise NotImplementedError("pooled mode needs feature planes that are a multiple of 8 pixels")
    if sp.xslab is None:
        sp.xslab = comm.symmetric(sp.x_bytes, dev)           # collective, first call only
    xs = sp.xslab
    par = xs.parity
    xs.parity ^= 1
    xo = sp.x_off[par]
    world, rank = comm.world, comm.rank
    ws = torch.empty(sp.ws_bytes, dtype=u8, device=dev)
    plan_dev = torch.empty(S * C.sizeof(_lib.ScalePlan), dtype=u8, device=dev)
    with _timed("sample"):
        # local histograms -> all-gather of the (image, class) counts -> identical global plan on every rank
        fn, fname = _plan_entry(lib, labels, hist_only=True)
        _lib.check(fn(C.byref(sp.cfg), labels.data_ptr(), ws.data_ptr(), st), fname)
        nA = sp.n_local * A
        local = torch.cat([ws[sp.counts_off[s]:sp.counts_off[s] + 4 * nA].view(i32) for s in range(S)])
        gathered = comm.all_gather(local).view(world, S, nA)
        counts_g = gathered.permute(1, 0, 2).contiguous()          # [S][n_global][A]
        cptr = _lib.ptr_array([counts_g[s].data_ptr() for s in range(S)])
        _lib.check(lib.mscs_sample_plan_from_counts(C.byref(sp.cfg), cptr, ws.data_ptr(), plan_dev.data_ptr(), st),
                   "mscs_sample_plan_from_counts")
        sizes = sp.slot_sizes
        islab = torch.empty(sp.islab_n, dtype=i32, device=dev)
        fslab = torch.empty(sp.fslab_n, dtype=f32, device=dev)
        misc = torch.empty(sp.misc_n, dtype=f32, device=dev)
        work = torch.empty(sp.work_bytes, dtype=u8, device=dev)
        slot_slab = torch.full((sum(sizes),), -1, dtype=i32, device=dev)
        slots, off = [], 0
        for x in sizes:
            slots.append(slot_slab[off:off + x])
            off += x
        # dense gradients (local): zero-filled on the side stream.  Row statistics: the sweeps accumulate them (one
        # atomic per row, quarter and tile) in PRIVATE memory; pushed to every rank's slab afterwards
        gradbufs = _GradBuffers(feats32, needs, False, 0) if any(needs) else None
        if gradbufs is not None:
            gradbufs.start_fill()
        stats_priv = torch.zeros(sp.stats_n, dtype=f32, device=dev)
        mt, pos = torch_mt_state()
        draws = _stream_cache(dev).acquire(mt, pos, sp.max_draws + _MT_N)
        plan = (_lib.ScalePlan * S)()
        ibase = islab.data_ptr()
        arrs = [_lib.ptr_array([ibase + 4 * sp.ioff[s][k] for s in range(S)]) for k in range(5)]
        sarr = _lib.ptr_array([x.data_ptr() for x in slots])
        fbase, bbase = fslab.data_ptr(), xs.local + xo["b"]
        # two views of the same terms: `job_sw` (sweeps: statistics in private memory) and `job` (finalise and
        # backward: statistics of ALL rows in the exchange slab)
        job, job_sw = _lib.SimJob(), _lib.SimJob()
        _fill_job(job, sp, A, bbase, ibase, xs.local + xo["stats"], misc.data_ptr(), work.data_ptr())
        _fill_job(job_sw, sp, A, bbase, ibase, stats_priv.data_ptr(), misc.data_ptr(), work.data_ptr())
        nt = len(sp.terms)
        mbase = misc.data_ptr()
        total_t = torch.empty((), dtype=f32, device=dev)      # own buffer, not a view (see _run_forward_fast)
        for jb in (job, job_sw):
            jb.term_loss, jb.total_loss = mbase + 4 * sp.out_off, mbase + 4 * (sp.out_off + nt)
            jb.total_out = total_t.data_ptr()
        # Selection and the peer-store gather are driven by the DEVICE plan records and enqueued before the host looks
        # at the plan: the one host wait of the forward (errors, row ranges) overlaps them instead of idling the GPU.
        device_driven = sp.v_cap * 12 <= 200 * 1024
        plan_sz = C.sizeof(_lib.ScalePlan)
        if device_driven:
            _lib.check(lib.mscs_plan_fetch_begin(plan_dev.data_ptr(), S, st), "mscs_plan_fetch_begin")
            _lib.check(lib.mscs_sample_select_async(C.byref(sp.cfg), plan_dev.data_ptr(), sp.v_cap, ws.data_ptr(),
                                                    draws.data_ptr(), *arrs, sarr, st), "mscs_sample_select_async")
        else:
            _lib.check(lib.mscs_plan_fetch(plan_dev.data_ptr(), plan, S, st), "mscs_plan_fetch")     # the host sync
            _raise_plan_errors(plan, S, spec)
            _lib.check(lib.mscs_sample_select(C.byref(sp.cfg), plan, ws.data_ptr(), draws.data_ptr(), *arrs, sarr, st),
                       "mscs_sample_select")
    with _timed("gather"):
        for s in range(S):
            n, Cc, h, w = sp.feat_shapes[s]
            _lib.check(lib.mscs_gather_normalize_p2p(
                feats32[s].data_ptr(), n, Cc, h * w, slots[s].data_ptr(), 0 if device_driven else plan[s].N,
                plan_dev.data_ptr() + s * plan_sz + 8 if device_driven else None, xs.peers, world, rank,
                xo["b"] + 2 * sp.boff[s], fbase + 4 * sp.foff[s][0], fbase + 4 * sp.foff[s][1], st),
                "mscs_gather_normalize_p2p")
        comm.barrier(xs)                                   # A: every rank's key rows have landed here
    if device_driven:
        _lib.check(lib.mscs_plan_fetch_end(plan, S), "mscs_plan_fetch_end")       # the host wait (plan records only)
        _raise_plan_errors(plan, S, spec)
    total = sum(int(plan[s].draws) for s in range(S))
    samples = [ScaleSample(plan[s].T, plan[s].V, plan[s].N, bool(plan[s].log_flag), plan[s].dl_h, plan[s].dl_w,
                           islab, sp.ioff[s], A) for s in range(S)]
    # this parity's gradient rows: only the 128-aligned row blocks this rank computes are accumulated into (and
    # pulled from): clear those (1/world of the slab), on the main stream, long before the backward
    if any(needs):
        zp, zb = [], []
        for s in range(S):
            rb, re_ = shard_rows(samples[s].N, world, rank)
            if re_ > rb:
                zp.append(xs.local + xo["dF"] + 4 * (sp.dF_off[s] + rb * sp.C_pad))
                zb.append(4 * ((re_ + 127) // 128 * 128 - rb) * sp.C_pad)
        if zp:
            _lib.check(lib.mscs_fill_bytes(_lib.ptr_array(zp), (C.c_int32 * len(zp))(*([0] * len(zp))),
                                           (C.c_size_t * len(zb))(*zb), len(zp), st), "mscs_fill_bytes")
    push_off, push_src, push_len = [], [], []
    for i, (a, k, *_rest) in enumerate(sp.terms):      # the plan-dependent fields of the jobs
        rb, re_ = shard_rows(samples[a].N, world, rank)      # anchor (and key) rows: sharded in 128-row granules
        kb, ke = shard_rows(samples[k].N, world, rank)
        for jb in (job, job_sw):
            t = jb.terms[i]
            t.N1, t.N2 = samples[a].N, samples[k].N
            t.row_begin, t.row_end, t.krow_begin, t.krow_end = rb, re_, kb, ke
        n1 = (sp.Ncap[a] + 15) // 16 * 16
        for q in range(3):      # neg, pos, S of this rank's rows
            push_src.append(sp.soff[i] + q * n1 + rb)
            push_off.append(xo["stats"] // 4 + sp.soff[i] + q * n1 + rb)
            push_len.append(re_ - rb)
    with _timed("sim_fwd"):
        _lib.check(lib.mscs_sim_forward_sweeps(C.byref(job_sw), st), "mscs_sim_forward_sweeps")
        _lib.check(lib.mscs_xchg_push(xs.peers, world, stats_priv.data_ptr(), (C.c_int64 * len(push_src))(*push_src),
                                      (C.c_int64 * len(push_off))(*push_off), (C.c_int32 * len(push_len))(*push_len),
                                      len(push_off), st), "mscs_xchg_push")
        comm.barrier(xs)                                   # B: the statistics of every row are complete here
        _lib.check(lib.mscs_sim_finalize(C.byref(job), st), "mscs_sim_finalize")
    if comm.owns_rng:
        _finish_rng(sp, dev, mt, pos, total)
    state = _StepState()
    state.sp, state.job, state.samples, state.gradbufs, state.slots = sp, job, samples, gradbufs, slots
    state.keep = (ws, islab, fslab, misc, work, slot_slab, stats_priv)
    state.stats = None
    state.fslab, state.term_loss = fslab, misc[sp.out_off:sp.out_off + nt]
    state.total = total_t
    state.scalars = misc[sp.out_off:sp.out_off + nt + 2]      # [term losses..., total, inf/NaN flag]: one copy for the logger
    state.num_ms, state.cs_logged, state.comm = S, sp.cs_logged, comm
    state.xs, state.par = xs, par
    n_local = sum(int(samples[s].N) for s in range(S)) / world        # rows this rank owns, on average
    state.exchange_info = {
        "transport": "NVLink peer stores / loads by the library's kernels (CUDA IPC slabs) + device-side flag barriers; "
                     "NCCL only for the class histograms",
        "barriers_per_step": 3,
        "nccl_all_gather_bytes": int(local.numel() * 4 * world),
        "key_rows_stored_to_peers_bytes": int(n_local * sp.C_pad * 2 * (world - 1)),
        "row_statistics_pushed_bytes": int(sum(push_len) * 4 * (world - 1)),
        "gradient_rows_pulled_bytes": int(n_local * sp.C_pad * 4 * (world - 1) / world)}
    return state


def _run_backward_pooled(state, grad_out, needs, shapes, dtypes):
    """Pooled mode: every rank computes the COMPLETE gradient rows of its 128-aligned row block of every anchor set
    (one launch for all passes) into its exchange slab; after the barrier the scatter pulls the row of every LOCAL
    pixel from the rank that computed it -- an eighth of the rows travels, once, to where it is needed."""
    lib = _lib.load()
    sp, comm, xs = state.sp, state.comm, state.xs
    dev, S = sp.dev, sp.S
    st = _stream()
    xo = sp.x_off[state.par]
    gb = state.gradbufs
    first = gb is not None and gb.ready is not None and not getattr(state, "bwd_done", False)
    if first:
        _cur_stream().wait_event(gb.ready)          # the side-stream zero fill (dense gradients + the slab's row region)
    else:                                           # second backward through the same graph: clear the row region again
        _lib.check(lib.mscs_fill_bytes(_lib.ptr_array([xs.local + xo["dF"]]), (C.c_int32 * 1)(0),
                                       (C.c_size_t * 1)(4 * sp.dF_n), 1, st), "mscs_fill_bytes")
        comm.barrier(xs)                            # nobody still pulls the previous rows
    state.bwd_done = True
    base = xs.local + xo["dF"]
    ptrs = [0] * _lib.MAX_SCALES
    lds = (C.c_int32 * _lib.MAX_SCALES)()
    for s in range(S):
        ptrs[s], lds[s] = base + 4 * sp.dF_off[s], sp.C_pad
    g = grad_out.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
    with _timed("sim_bwd"):
        _lib.check(lib.mscs_sim_backward(C.byref(state.job), g.data_ptr(), _lib.ptr_array(ptrs), lds, st),
                   "mscs_sim_backward")
        comm.barrier(xs)                            # C: every rank's gradient rows are complete
    grads = []
    fbase = state.fslab.data_ptr()
    with _timed("scatter"):
        for s in range(S):
            if not needs[s]:
                grads.append(None)
                continue
            n, Cc, h, w = shapes[s]
            pre = gb.take(s) if gb is not None else None
            if pre is None:
                pre = torch.zeros(shapes[s], dtype=torch.float32, device=dev)
            N = state.samples[s].N
            per = ((N + 127) // 128 + comm.world - 1) // comm.world * 128
            _lib.check(lib.mscs_scatter_sectors_pull(xs.peers, comm.world, xo["dF"] + 4 * sp.dF_off[s], per, sp.C_pad,
                                                     fbase + 4 * sp.foff[s][0], fbase + 4 * sp.foff[s][1],
                                                     state.slots[s].data_ptr(), n, Cc, h * w, pre.data_ptr(), st),
                       "mscs_scatter_sectors_pull")
            grads.append(pre if dtypes[s] == torch.float32 else pre.to(dtypes[s]))
    return grads


def run_backward(state, grad_out, needs, shapes, dtypes):
    lib = _lib.load()
    sp = state.sp
    dev, S = sp.dev, sp.S
    st = _stream()
    if state.comm is not None:
        return _run_backward_pooled(state, grad_out, needs, shapes, dtypes)
    # gradient-row accumulators: cleared during the forward -- inside the workspace by the sampling chain's fills
    # (default), or together with the pre-zeroed dense gradients on the side stream; a second backward through the
    # same graph takes a fresh zeroed buffer
    dF, base, e = None, None, getattr(state, "entry", None)
    first = not getattr(state, "bwd_done", False)
    state.bwd_done = True
    if state.gradbufs is not None:
        dF = state.gradbufs.take_dF()
        if dF is not None:
            _cur_stream().wait_event(state.gradbufs.ready)
    elif first and getattr(state, "dF_ws", None):
        base = state.dF_ws
    in_ws = base is not None
    if not in_ws:
        if dF is None:
            dF = torch.zeros(sp.dF_n, dtype=torch.float32, device=dev)
        base = dF.data_ptr()
    if in_ws:
        ptrs_arr, lds = e.bw_ptrs, e.bw_lds
        ptrs = [base + 4 * sp.dF_off[s] for s in range(S)]
    else:
        ptrs = [0] * _lib.MAX_SCALES
        lds = (C.c_int32 * _lib.MAX_SCALES)()
        for s in range(S):
            ptrs[s], lds[s] = base + 4 * sp.dF_off[s], sp.C_pad
        ptrs_arr = _lib.ptr_array(ptrs)
    if grad_out.dtype == torch.float32 and grad_out.device == dev and grad_out.is_contiguous():
        g = grad_out                      # (only its address is used)
    else:
        g = grad_out.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
    grads = []
    fbase = state.fslab.data_ptr()
    io = state.io_dtypes or [torch.float32] * S         # dtypes the kernels write the dense gradients in
    # a captured call: row counts only on the device (upper bounds on the host), no generator prefetch to launch
    graph = getattr(state, "graph", False)
    rows_dev = e.rows_dev if graph else [None] * S
    n_rows = (lambda s: sp.Ncap[s]) if graph else (lambda s: state.samples[s].N)
    dense = (not sp.nhwc) and state.gradbufs is None and \
        all((not needs[s]) or (state.slots[s] is not None) for s in range(S))
    if dense:
        # default path: similarity backward + normalisation backward + one-pass dense writer in ONE C call
        idx = [s for s in range(S) if needs[s]]
        pre = getattr(state, "grad_slab", None) if (in_ws and len(idx) == S) else None
        if pre is not None:                 # allocated and entered into the prebuilt structures by the forward
            state.grad_slab = None
            slab, items, rows = pre, e.bw_items, e.bw_rows
            outs = dict(enumerate(state.grad_outs))
            state.grad_outs = None
        else:
            slab, views, offs = _dense_grad_slab([shapes[s] for s in idx], [io[s] for s in idx], dev)
            sbase = slab.data_ptr()
            outs = {}
            items = (_lib.ScatterItem * max(1, len(idx)))()
            rows = (C.c_int32 * max(1, len(idx)))()
            for j, s in enumerate(idx):
                n, Cc, h, w = shapes[s]
                outs[s] = views[j]
                it = items[j]
                it.dF, it.ldF, it.anc_f32, it.inv_norm = ptrs[s], sp.C_pad, fbase + 4 * sp.foff[s][0], fbase + 4 * sp.foff[s][1]
                it.slot, it.n, it.C, it.plane = state.slots[s].data_ptr(), n, Cc, h * w
                it.dfeat, it.dtype, it.n_rows_dev = sbase + offs[j], _DTYPE_CODE[io[s]], rows_dev[s]
                rows[j] = n_rows(s)
        evs, evp = None, None
        if TIMING is not None:
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(3 if TIMING_ALL else 2)]
            for ev in evs:
                ev.record()         # creates the CUDA event; the chain records it again at its stage boundary
            evp = _lib.ptr_array([ev.cuda_event for ev in evs] + [None] * (3 - len(evs)))
        _lib.check(lib.mscs_backward_chain(C.byref(state.job), g.data_ptr(), ptrs_arr, lds, items, rows,
                                           len(idx), evp, st), "mscs_backward_chain")
        if not graph:
            _stream_cache(dev).flush()    # the deferred generator launch of the next call's stream
        if evs is not None:
            TIMING.setdefault("sim_bwd", []).append((evs[0], evs[1]))
            if len(evs) == 3:
                TIMING.setdefault("scatter", []).append((evs[1], evs[2]))
        return [None if not needs[s] else (outs[s] if outs[s].dtype == dtypes[s] else outs[s].to(dtypes[s]))
                for s in range(S)]
    with _timed("sim_bwd"):
        _lib.check(lib.mscs_sim_backward(C.byref(state.job), g.data_ptr(), ptrs_arr, lds, st),
                   "mscs_sim_backward")
    if not graph:
        _stream_cache(dev).flush()        # the deferred generator launch of the next call's stream
    if sp.nhwc:
        with _timed("scatter"):
            gb = state.gradbufs
            if gb is not None:
                _cur_stream().wait_event(gb.ready)
            idx = [s for s in range(S) if needs[s]]
            items = (_lib.RowsItem * max(1, len(idx)))()
            outs = {}
            for j, s in enumerate(idx):
                n, Cc, h, w = shapes[s]
                pre = gb.take(s) if gb is not None else None
                if pre is None:      # second backward through the same graph
                    pre = torch.zeros((n, h, w, Cc), dtype=io[s], device=dev).permute(0, 3, 1, 2)
                outs[s] = pre
                it = items[j]
                it.pix = e.islab.data_ptr() + 4 * sp.ioff[s][2] if graph else state.samples[s].ptr(2)
                it.rows, it.C, it.n_rows_dev = n_rows(s), Cc, rows_dev[s]
                it.anc_f32, it.inv_norm = fbase + 4 * sp.foff[s][0], fbase + 4 * sp.foff[s][1]
                it.dF, it.ldF, it.dfeat, it.dtype = ptrs[s], sp.C_pad, pre.data_ptr(), _DTYPE_CODE[io[s]]
            if idx:
                _lib.check(lib.mscs_scatter_rows_nhwc_batch(items, len(idx), st), "mscs_scatter_rows_nhwc_batch")
            return [None if not needs[s] else (outs[s] if outs[s].dtype == dtypes[s] else outs[s].to(dtypes[s]))
                    for s in range(S)]
    with _timed("scatter"):
        gb = state.gradbufs
        if gb is not None:
            _cur_stream().wait_event(gb.ready)
        batch = []
        for s in range(S):
            if not needs[s]:
                grads.append(None)
                continue
            n, Cc, h, w = shapes[s]
            smp = state.samples[s]
            pre, slot = (gb.take(s) if gb is not None else None), state.slots[s]
            if pre is not None and slot is not None:
                out = pre
                # every scale in one launch (below)
                batch.append((ptrs[s], fbase + 4 * sp.foff[s][0], fbase + 4 * sp.foff[s][1], slot.data_ptr(),
                              n, Cc, h * w, out.data_ptr()))
            else:
                out = torch.empty(shapes[s], dtype=torch.float32, device=dev)
                _lib.check(lib.mscs_scatter_grad(ptrs[s], sp.C_pad, fbase + 4 * sp.foff[s][0],
                                                 fbase + 4 * sp.foff[s][1], smp.ptr(2), smp.N, n, Cc, h * w,
                                                 out.data_ptr(), 1, st), "mscs_scatter_grad")
            grads.append(out)
        if batch:
            items = (_lib.ScatterItem * len(batch))()
            for it, (dfp, f32p, invp, slotp, n, Cc, plane, outp) in zip(items, batch):
                it.dF, it.ldF, it.anc_f32, it.inv_norm, it.slot = dfp, sp.C_pad, f32p, invp, slotp
                it.n, it.C, it.plane, it.dfeat = n, Cc, plane, outp
            _lib.check(lib.mscs_scatter_sectors_batch(items, len(batch), st), "mscs_scatter_sectors_batch")
        grads = [g_ if (g_ is None or dtypes[s] == torch.float32) else g_.to(dtypes[s]) for s, g_ in enumerate(grads)]
    return grads


# ---- the autograd.Function ----------------------------------------------------------------
_device_checked = [False]


class MsCsContrastiveFn(torch.autograd.Function):
    """(labels, spec, single_scale, holder, *features) -> (total_loss 0-d, term_losses (n_terms,)).

    ``holder`` (a dict) receives the sampling results and term bookkeeping for the caller
    (log_this_step, ms/cs split, reference-order indices)."""

    @staticmethod
    def forward(ctx, labels, spec, single_scale, holder, *feats):
        comm = holder.get("comm")
        world = comm.world if comm is not None else 1
        philox = holder.get("philox")
        # decided (and refused) before anything is enqueued
        graph = graph_mode(spec, world, single_scale, labels, feats, philox[1] if philox is not None else None)
        if not _device_checked[0]:
            if not _lib.load().mscs_device_ok():
                raise RuntimeError("mscs_b200 needs a compute-capability 10.x (B200) device; no fallback exists")
            _device_checked[0] = True
        # channels-last feature maps (memory order [n][h][w][C]) are consumed as they are by the single-process fast
        # path: an anchor is then one contiguous row (gather / scatter become row copies)
        nhwc = channels_last_ok(spec, world, feats)
        for f in feats:
            _require_device(f)
        dev = feats[0].device
        if labels.device != dev:
            labels = labels.to(dev)
        needs = [bool(ctx.needs_input_grad[4 + i]) for i in range(len(feats))]
        if labels.dtype not in (torch.int64, torch.int16):     # int16: compact labels of the fused label pass
            labels = labels.long()
        labels = labels.contiguous()
        with torch.cuda.device(dev), _pin_stream():
            world, rank = (comm.world, comm.rank) if comm is not None else (1, 0)
            sp = _step_plan(dev, labels.shape, [tuple(f.shape) for f in feats], spec, single_scale, world, rank, nhwc)
            # bf16 / fp16 maps go to the kernels as they are where half_io_ok holds; everything else as an fp32 copy
            half_ok = half_io_ok(sp, world)
            maps = []
            for f in feats:
                m = f.detach()
                if m.dtype != torch.float32 and not (half_ok and m.dtype in _DTYPE_CODE):
                    m = m.float()
                maps.append(m if nhwc else m.contiguous())
            state = run_forward(sp, labels, maps, needs, comm, philox, graph)
        holder["samples"], holder["state"] = state.samples, state
        ctx.state, ctx.needs = state, needs
        ctx.shapes = [tuple(f.shape) for f in feats]
        ctx.dtypes = [f.dtype for f in feats]
        # 0-d tensor with storage of its own: tolerates the caller's `loss *= w`.  The state must NOT keep it: an output
        # of this Function references its grad_fn, which owns ctx.state -- a cycle through C++ that Python's collector
        # cannot see (the state, its workspace and the dense-gradient slab would never be returned)
        total, state.total = state.total, None
        terms = state.term_loss
        ctx.mark_non_differentiable(terms)
        ctx.set_materialize_grads(False)       # no zero tensor (a fill launch) for the unused gradient of `terms`
        return total, terms

    @staticmethod
    def backward(ctx, grad_total, _grad_terms):
        if grad_total is None:
            return (None,) * (4 + len(ctx.needs))
        with torch.cuda.device(ctx.state.sp.dev), _pin_stream():
            grads = run_backward(ctx.state, grad_total, ctx.needs, ctx.shapes, ctx.dtypes)
        return (None, None, None, None, *grads)
