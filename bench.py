#!/usr/bin/env python
"""Benchmark of the ms+cs dense contrastive loss hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2] [--dump-outputs DIR]

A step = one forward + backward of the loss over one batch of synthetic inputs (SURVEY.md §8d).
N=1 workload: cfg2 = HRNet-W48 Cityscapes ms+cs (4 scales, 512x1024 crops, bs 12, 256-d).
N>1: one process per GPU, every rank runs the same per-GPU workload on its own batch (what the
reference does under DDP: the loss is evaluated per rank on the local mini-batch, no collective on
this path) -> weak scaling; value = anchor-pairs of all ranks / max-over-ranks device time.
`--workload cfg5` is the POOLED cross-batch configuration instead (64 images in total, anchor rows
sharded over the ranks, keys exchanged over NCCL): total work fixed -> strong scaling.

Prints ONE JSON line (rank 0).  `--impl reference` times the reference's own implementation on the host cores: the
unmodified loss files staged under oracle/_ref/ (oracle/make_ref.py; /root/reference does not exist on the GPU box),
or, if those are absent, the fp32 torch port of the oracle (oracle/torch_port.py).
Defaults: K=100 timed steps after W=20 warm-up steps (a step is ~1 ms; the short 20/5 default of the first
versions made the timed region sensitive to the start-up of a fresh process); `--impl reference`: K=5, W=1 (a CPU
step takes seconds); exactly K steps after W are timed on a bounded SAMPLE of the workload (the first images of the same
batch), sized from a calibration step so that the run ends within ~4 minutes (`cpu_baseline.sample` says which).
--steps / --warmup set the timed loop of the headline number; the two side records of the GPU run keep fixed counts,
stated in their own fields: `pooled` (cfg5, 10 steps after 3) and `cpu_baseline` (2 steps after 1 on 3 images).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC, UNIT = "ms+cs contrastive loss fwd+bwd anchor-pairs/s", "anchor-pairs/s"
# bounded CPU sample of the workload: the first CPU_SAMPLE_IMAGES images of the same inputs (3 = the
# per-rank batch of the reference's own 4-GPU recipe, README.md:51); one step is a few seconds
CPU_SAMPLE_IMAGES = 3


def pairs_per_step(NS, cross_scale):
    """sum over terms of N_a * N_k (SURVEY.md §8d)."""
    p = sum(n * n for n in NS)
    if cross_scale and len(NS) > 1:
        p += NS[0] * NS[-1]
        if len(NS) > 2:
            p += NS[0] * NS[-2]
    return p


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(tflops=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained") or d["bf16_tflops"],
                    hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock and throttle reasons sampled every 100 ms during the timed region (NVML in-process:
    an external `nvidia-smi -lms` loop perturbs sub-second timed regions)."""

    def __init__(self, index):
        self.rows, self.index, self.stop_flag, self.thread, self.h = [], index, False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nv = None

    def _sample(self):
        nv = self.nv
        return (nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))

    def _loop(self):
        while not self.stop_flag:
            try:
                self.rows.append(self._sample())
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        if self.nv is None:
            return
        self.rows.append(self._sample())
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join()
        self.rows.append(self._sample())
        nv = self.nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM),
                "reasons": sorted(k for k, v in names.items() if bits & v), "samples": len(sm)}


def _ref_modules():
    """The reference's own loss classes (oracle/_ref or /root/reference, unmodified; `.cuda()` neutralised so that they
    run on the host cores), or None when the staged files are absent -- then the torch port of the oracle is timed."""
    try:
        from oracle import ref_loader
        return ref_loader.load(cpu=True)
    except FileNotFoundError:
        return None


def cpu_step(ref, cfg, ocfg, labels, feats, torch_port):
    """One forward + backward of the loss on the host: the reference classes themselves (kind "reference") or the
    fp32 torch port of the oracle (kind "port")."""
    fg = [f.clone().requires_grad_(True) for f in feats]
    t0 = time.perf_counter()
    if ref is not None:
        if cfg["single_scale"]:
            total = ref.DenseContrastiveLossV2(dict(cfg["loss"]))(labels, fg[0])
        else:
            total = ref.DenseContrastiveLossV2_ms(dict(cfg["loss"]))(labels, fg)
    else:
        total = torch_port.ms_cs_loss(labels, fg, ocfg)[0]
    total.backward()
    return time.perf_counter() - t0, float(total.detach())


def anchors_per_scale(labels, feats, ocfg):
    """N per scale of a batch (a function of the labels and the caps only): from the sampling oracle."""
    from oracle.sampling import sample_indices
    from oracle.mt19937 import MT19937
    gen = MT19937.from_torch_state(torch.get_rng_state().numpy().tobytes())
    out = []
    for f in feats:
        o = sample_indices(labels.numpy(), f.shape[-1], ocfg["num_all_classes"], ocfg["min_views"], ocfg["max_views"],
                           ocfg["max_total"], gen)
        out.append(int(o["T"]) * int(o["V"]))
    return out


def cpu_sample(workload, steps, warmup, budget_s, images=None):
    """The reference loss timed on the host cores on a bounded sample of the workload: the first `images` images of
    the same inputs.  images=None: the largest of (all, half, quarter, ...) whose (warmup + steps) steps fit the
    time budget, estimated from one calibration step on the smallest sample."""
    from mscs_b200 import synth
    from oracle import torch_port
    from oracle.config import oracle_cfg
    from mscs_b200.datasets import class_facts
    cfg = synth.CONFIGS[workload]
    lc = dict(cfg["loss"])
    ocfg = oracle_cfg(lc, class_facts(lc["dataset"], lc["experiment"])[0])
    if cfg["single_scale"]:
        ocfg["cross_scale"], ocfg["weights"] = False, [1.0]
    ref = _ref_modules()
    labels_all, feats_all = synth.make_inputs(workload)
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    n_all = labels_all.shape[0]

    def subset(k):
        return labels_all[:k].contiguous(), [f[:k].contiguous() for f in feats_all]

    t_begin = time.perf_counter()
    calib = ""
    if images is None:
        small = min(CPU_SAMPLE_IMAGES, n_all)
        lab, fts = subset(small)
        torch.manual_seed(0)
        cpu_step(ref, cfg, ocfg, lab, fts, torch_port)               # untimed: thread pool, allocator, imports
        torch.manual_seed(1)
        t_small, _ = cpu_step(ref, cfg, ocfg, lab, fts, torch_port)
        images = small
        k = n_all
        while k > small:        # measured: the step time grows like images^1.3 (the per-pair dense scatter backward)
            if (warmup + steps) * t_small * (k / small) ** 1.3 <= budget_s - (time.perf_counter() - t_begin):
                images = k
                break
            k //= 2
        calib = f"; sample sized by a calibration step ({t_small:.1f} s at {small} images) for a {budget_s:.0f} s budget"
    labels, feats = subset(images)
    torch.manual_seed(0)
    NS = anchors_per_scale(labels, feats, ocfg)
    times = []
    for i in range(warmup + steps):
        torch.manual_seed(i)
        dt, _ = cpu_step(ref, cfg, ocfg, labels, feats, torch_port)
        if i >= warmup:
            times.append(dt)
    pairs = pairs_per_step(NS, ocfg["cross_scale"])
    sec = sum(times) / len(times)
    kind = "reference" if ref is not None else "port"
    what = ("the reference's own losses/DenseContrastiveLossV2_ms.py + DenseContrastiveLossV2.py (unmodified, "
            "oracle/_ref), fp32 ATen on the host") if ref is not None else "oracle/torch_port.py (fp32 torch port)"
    return dict(value=pairs / sec, unit=UNIT, cores=cores, kind=kind,
                sample=f"first {images} of {n_all} images of the {workload} inputs (N per scale {NS}, {pairs:.3e} "
                       f"anchor-pairs/step; N is bound by max_features_total, so the work per step is that of the "
                       f"full batch to within a few percent), {len(times)} timed steps after {warmup} warm-up; {what}, "
                       f"torch {torch.__version__}, {torch.get_num_threads()} threads{calib}",
                seconds_per_step=sec, pairs_per_step=pairs, steps_timed=len(times))


def workload_name(workload):
    """`config.workload` of the JSON line -- the same string on both arms (the driver pairs the lines by it)."""
    return f"{workload}: " + {
        "cfg2": "HRNet-W48 Cityscapes ms+cs loss, 4 scales, 512x1024 crops, bs 12, 256-d projector",
        "cfg5": "pooled cross-batch anchors, bs 64 in total, ms+cs, max_features_total 65536"}.get(workload, workload)


def bench_config(workload, world, layout="nchw"):
    """`config` of the JSON line: the same dict on both arms (the driver pairs the two lines by it)."""
    from mscs_b200 import synth
    cfg = synth.CONFIGS[workload]
    feat_mb = sum(cfg["n"] * cfg["C"] * (cfg["H"] // s) * (cfg["W"] // s) * 4 for s in cfg["strides"]) / 1e6
    pooled = workload == "cfg5"
    return {"workload": workload_name(workload), "layout": layout,
            "per_gpu_batch": cfg["n"] // world if pooled else cfg["n"],
            "l2": f"inputs ({feat_mb:.0f} MB of features per step) exceed the 126 MB L2; no explicit flush",
            "parallelism": (f"pooled anchors: rows sharded x{world}, keys / row statistics / gradient rows exchanged "
                            f"over NCCL" if pooled else
                            f"replicas x{world} (loss evaluated per rank on its local batch, as under DDP)")}


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path on the host cores (oracle/_ref = the unmodified files), on a
    bounded sample of the same workload: exactly --steps timed steps after --warmup, the sample (number of images)
    sized so that the run ends within ~4 minutes.  Rank 0 only."""
    if rank != 0:
        return
    cb = cpu_sample(args.workload, args.steps, args.warmup, budget_s=240.0)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": cb["steps_timed"], "warmup": args.warmup, "ms_per_step": cb["seconds_per_step"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args.workload, args.gpus),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, loss, mod, feats):
    """Writes what one step returned to its caller as ``out_dir/<name>.npy``: ``loss``, the per-scale terms the module
    exposes for logging (``ms_losses``, ``cs_losses``), and per scale the dense feature gradient at the pixels that
    carry one (every other entry is exactly zero): ``grad<s>_pixels`` (flat index (image * h + y) * w + x, float64) and
    ``grad<s>_rows`` (pixels x C, float32).  A scale whose rows exceed its share of DUMP_BYTES keeps a fixed, seeded
    sample of them (pixel order kept)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": np.array([float(loss.detach())], dtype=np.float64)}
    for key in ("ms_losses", "cs_losses"):
        vals = getattr(mod, key, None)
        if vals:
            arrays[key] = np.array([float(v) for v in vals], dtype=np.float64)
    share = (DUMP_BYTES - (1 << 20)) // len(feats)
    for s, f in enumerate(feats):
        C = f.shape[1]
        g = f.grad.detach().permute(0, 2, 3, 1).reshape(-1, C)
        pix = (g != 0).any(dim=1).nonzero().squeeze(1)
        keep = share // (C * 4 + 8)
        if pix.numel() > keep:
            sel = torch.randperm(pix.numel(), generator=torch.Generator().manual_seed(s))[:keep].sort().values
            pix = pix[sel.to(pix.device)]
        arrays[f"grad{s}_pixels"] = pix.cpu().double().numpy()
        arrays[f"grad{s}_rows"] = g[pix].float().cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_pooled(dev, rank, world, dist, steps=10, warmup=3):
    """The sharded configuration north_star names (cfg5: 64 images pooled over the ranks, anchor rows sharded, keys /
    row statistics / gradient rows exchanged): ms per step at this world size and -- measured in the same run by rank 0
    alone on the full batch -- the single-GPU time it is compared with (strong scaling).  Labels are the cfg5 labels
    (same (T, V) as the parity fixtures); features are drawn on the device per (scale, image), identical for every
    world size."""
    import mscs_b200
    from mscs_b200 import synth
    cfg = synth.CONFIGS["cfg5"]
    labels_all = synth.make_labels(cfg)
    n = cfg["n"]

    def inputs(i0, i1):
        fts = []
        for si, st in enumerate(cfg["strides"]):
            f = torch.empty((i1 - i0, cfg["C"], cfg["H"] // st, cfg["W"] // st), device=dev)
            for b in range(i0, i1):
                g = torch.Generator(device=dev)
                g.manual_seed(100003 * (si + 1) + b)
                f[b - i0].normal_(generator=g)
            fts.append(f.requires_grad_(True))
        return labels_all[i0:i1].contiguous().to(dev), fts

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run(comm, lab, fts, sync):
        mod = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg["loss"]), comm=comm) if comm is not None else \
            mscs_b200.DenseContrastiveLossV2_ms(dict(cfg["loss"]))
        torch.manual_seed(0)                 # every rank: same CPU generator state (the pooled plan consumes it)

        def one():
            for f in fts:
                f.grad = None
            loss = mod(lab, fts)
            loss.backward()
            return loss
        for _ in range(warmup):
            one()
        from mscs_b200 import _ops
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync()
        e0.record()
        for _ in range(steps):
            loss = one()
        e1.record()
        sync()
        # stage breakdown: a second pass (the stage events are not part of the product path and cost ~50 us per step)
        _ops.TIMING, _ops.TIMING_ALL = {}, True
        for _ in range(max(3, steps // 2)):
            one()
        sync()
        mod.stage_ms = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in _ops.TIMING.items()}
        _ops.TIMING = None
        NS = [s_.N for s_ in mod.last_samples]
        return e0.elapsed_time(e1) / steps, float(loss.detach()), NS, mod

    out = {"workload": workload_name("cfg5"), "n_gpus": world, "steps": steps, "warmup": warmup, "scaling": "strong"}
    single_ms = None
    if rank == 0:        # the single-GPU reference time of the same batch (the other ranks wait at the barrier below)
        lab, fts = inputs(0, n)
        single_ms, loss1, NS, _m = run(None, lab, fts, torch.cuda.synchronize)
        out.update(single_gpu_ms_per_step=single_ms, single_gpu_loss=loss1, anchors_per_scale=NS,
                   single_gpu_stage_ms=_m.stage_ms)
        del lab, fts, _m
        torch.cuda.empty_cache()
    if world > 1:
        barrier()
        nl = n // world
        lab, fts = inputs(rank * nl, (rank + 1) * nl)
        ms, loss, NS, mod = run(mscs_b200.TorchDistComm(), lab, fts, barrier)
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
        if rank == 0:
            pairs = pairs_per_step(NS, True)
            out.update(ms_per_step=ms, value=pairs / (ms * 1e-3), unit=UNIT, loss=loss, stage_ms_rank0=mod.stage_ms,
                       speedup_vs_single_gpu=single_ms / ms, efficiency=single_ms / ms / world,
                       exchange=mod.last_state.exchange_info if hasattr(mod.last_state, "exchange_info") else None)
    elif rank == 0:
        pairs = pairs_per_step(out["anchors_per_scale"], True)
        out.update(ms_per_step=single_ms, value=pairs / (single_ms * 1e-3), unit=UNIT)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # a step is ~1 ms: the defaults keep the timed region (0.1 s) well above start-up effects of a fresh process
    # (cold page cache, allocator growth); the whole default run still takes well under a minute
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of the headline loop; default: 100 (--impl reference: 5). The pooled and "
                         "cpu_baseline side records use fixed counts (see the module docstring)")
    ap.add_argument("--warmup", type=int, default=None, help="default: 20 (--impl reference: 1)")
    ap.add_argument("--impl", default="mscs", choices=["mscs", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pooled", action="store_true", help="skip the cfg5 (pooled, sharded) record")
    ap.add_argument("--layout", default="nchw", choices=["nchw", "nhwc"],
                    help="memory order of the feature maps: nchw = what the reference's projector emits (headline); "
                         "nhwc = torch.channels_last (row gather / scatter)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss, its logged per-scale terms and the feature gradients "
                         "of the last timed step as DIR/<name>.npy (rank 0; at most 64 MB, see dump_outputs)")
    args = ap.parse_args()
    ref = args.impl == "reference"       # a reference step is seconds of CPU work, one of ours a millisecond
    if ref and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the GPU path; it does not apply to --impl reference")
    args.steps = args.steps if args.steps is not None else (5 if ref else 100)
    args.warmup = args.warmup if args.warmup is not None else (1 if ref else 20)
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import mscs_b200
    from mscs_b200 import _ops, synth
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists)"
    args.warmup = max(args.warmup, 3)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    cfg = synth.CONFIGS[args.workload]
    labels_h, feats_h = synth.make_inputs(args.workload)
    pooled = args.workload == "cfg5"
    comm = None
    if pooled and world > 1:        # every rank owns a contiguous block of the 64 images
        nl = cfg["n"] // world
        labels_h = labels_h[rank * nl:(rank + 1) * nl].contiguous()
        feats_h = [f[rank * nl:(rank + 1) * nl].contiguous() for f in feats_h]
        comm = mscs_b200.TorchDistComm()
    labels_h = labels_h.pin_memory()
    if args.layout == "nhwc":       # pinned [n][h][w][C] storage viewed as (n, C, h, w)
        feats_h = [torch.empty((f.shape[0], f.shape[2], f.shape[3], f.shape[1]), pin_memory=True)
                   .permute(0, 3, 1, 2).copy_(f) for f in feats_h]
    else:
        feats_h = [f.pin_memory() for f in feats_h]
    cls = mscs_b200.DenseContrastiveLossV2 if cfg["single_scale"] else mscs_b200.DenseContrastiveLossV2_ms
    mod = cls(dict(cfg["loss"]), comm=comm) if comm is not None else cls(dict(cfg["loss"]))
    labels = labels_h.to(dev)
    feats = [f.to(dev).requires_grad_(True) for f in feats_h]
    if args.layout == "nhwc":
        assert all(f.is_contiguous(memory_format=torch.channels_last) and not f.is_contiguous() for f in feats)

    torch.manual_seed(0)      # seeded once, like a training run: the generator then only advances

    def step(lab, fts, seed):
        for f in fts:
            f.grad = None
        loss = mod(lab, fts[0] if cfg["single_scale"] else fts)
        loss.backward()
        return loss

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing -----------------------------------------------------------
    for i in range(args.warmup):
        step(labels, feats, i)
    NS = [s.N for s in mod.last_samples]
    assert mod.last_state.sp.nhwc == (args.layout == "nhwc"), "feature layout did not select the expected kernels"
    pairs = pairs_per_step(NS, mod._spec.cross_scale and not cfg["single_scale"])
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the DOMINANT kernel (k_sim_bwd) is bracketed by CUDA events INSIDE the timed region, on the launching stream: the
    # duration behind the roofline is that of the sustained loop, not of a cold burst.  The other stages are timed in a
    # second pass right after it: a full set of stage events costs ~50 us per step (16 records, which also sit between
    # kernels that otherwise overlap through programmatic dependent launch), and that is not part of the product path.
    _ops.TIMING, _ops.TIMING_ALL = {}, False
    e0.record()
    for i in range(args.steps):
        loss = step(labels, feats, 100 + i)
    e1.record()
    barrier()
    stage_ms = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in _ops.TIMING.items()}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, mod, feats)
    _ops.TIMING, _ops.TIMING_ALL = {}, True
    n_stage = max(3, min(args.steps, 50))
    for i in range(n_stage):
        step(labels, feats, 5000 + i)
    barrier()
    stage_all = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in _ops.TIMING.items()}
    stage_all["sim_bwd_second_pass"] = stage_all["sim_bwd"]
    stage_ms = {**stage_all, **stage_ms}        # sim_bwd: from the timed region
    _ops.TIMING = None
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms) / args.steps
    share = 1 if pooled else world       # pooled: `pairs` already is the whole job
    value = pairs * share / (ms_step * 1e-3)

    # ---- end to end through the public API with HOST buffers -------------------------------
    h2d = labels_h.numel() * 8 + sum(f.numel() * 4 for f in feats_h)
    d2h = 4

    def e2e_step(seed):
        lab = labels_h.to(dev, non_blocking=True)
        fts = [f.to(dev, non_blocking=True).requires_grad_(True) for f in feats_h]
        return float(step(lab, fts, seed).detach().cpu())       # D2H read of the loss (synchronises)

    copy_st = torch.cuda.Stream(device=dev)

    def stage_inputs():
        """H2D copy of ONE step's inputs from pinned host memory, on the copy stream."""
        with torch.cuda.stream(copy_st):
            lab = labels_h.to(dev, non_blocking=True)
            fts = [f.to(dev, non_blocking=True) for f in feats_h]
            ev = torch.cuda.Event()
            ev.record(copy_st)
        return lab, fts, ev

    def e2e_pipelined(n):
        """Every step copies its own inputs from the host and reads its loss back; the copy of step i+1 is issued
        before step i's kernels (double buffering, what a prefetching loader does), so it overlaps them."""
        cur = torch.cuda.current_stream()
        nxt = stage_inputs()
        out = 0.0
        for i in range(n):
            lab, fts, ev = nxt
            if i + 1 < n:
                nxt = stage_inputs()
            cur.wait_event(ev)
            for t in [lab] + fts:
                t.record_stream(cur)
            out = float(step(lab, [f.requires_grad_(True) for f in fts], i).detach().cpu())   # D2H read of the loss
        return out

    def timed(fn):
        barrier()
        e0.record()
        fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    n_e2e = max(3, min(args.steps // 2, 40))
    for i in range(3):
        e2e_step(i)
    e2e_serial_ms = timed(lambda: [e2e_step(200 + i) for i in range(n_e2e)]) / n_e2e
    e2e_pipelined(3)
    e2e_ms = timed(lambda: e2e_pipelined(n_e2e)) / n_e2e
    e2e_val = pairs * share / (e2e_ms * 1e-3)

    # ---- roofline of the dominant kernel from the per-stage device times of the timed loop
    pk = peaks()
    Cdim = cfg["C"]
    per_gpu = pairs / world if pooled else pairs
    bwd_flops = 4.0 * Cdim * per_gpu          # K4: two gradient products per anchor pair (SURVEY.md §8d)
    fwd_flops = 2.0 * Cdim * per_gpu
    t_bwd = stage_ms.get("sim_bwd", float("nan")) * 1e-3
    achieved = bwd_flops / t_bwd / 1e12
    # DRAM traffic of one k_sim_bwd launch at cfg-2: a CONSTANT copied from the ncu --set full capture summarised in
    # profiles/ (dram__bytes_read.sum + dram__bytes_write.sum), not measured by this run; other workloads: not captured
    traffic = 51.0e6 + 0.06e6 if (args.workload == "cfg2" and not pooled) else None
    # Denominator: the BURST cuBLAS bf16 figure of MEASURED_PEAKS.json.  The timed region of the default run is a
    # fraction of a second at full SM clock, so the sustained (power-limited, 4 s) figure would flatter the kernel.
    roofline = {"bound": "tensor", "kernel": "k_sim_bwd", "achieved": achieved, "peak": pk["tflops"],
                "unit": "TFLOP/s", "frac": achieved / pk["tflops"], "traffic": traffic,
                "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum; constant from the "
                                "committed capture in profiles/, not re-measured here)",
                "peak_source": pk["source"] + ": burst cuBLAS bf16 (sustained figure %.1f)" % pk["tflops_sustained"],
                "frac_of_sustained_peak": achieved / pk["tflops_sustained"],
                "algorithmic_flops_per_launch": bwd_flops,
                "launch_ms": t_bwd * 1e3,
                "fwd": {"kernel": "k_sim_fwd (2 sweeps + row ranges, work tables, finalise)",
                        "achieved": fwd_flops / (stage_ms["sim_fwd"] * 1e-3) / 1e12,
                        "frac": fwd_flops / (stage_ms["sim_fwd"] * 1e-3) / 1e12 / pk["tflops"],
                        "launch_ms": stage_ms["sim_fwd"]},
                "similarity_kernels": {"achieved": (fwd_flops + bwd_flops) / ((stage_ms["sim_fwd"] + stage_ms["sim_bwd"])
                                                                               * 1e-3) / 1e12,
                                       "frac": (fwd_flops + bwd_flops) / ((stage_ms["sim_fwd"] + stage_ms["sim_bwd"])
                                                                          * 1e-3) / 1e12 / pk["tflops"]},
                "stage_ms": stage_ms,
                "stage_ms_note": "sim_bwd: CUDA events inside the timed region; the other stages: a second pass of %d "
                                 "steps right after it with the full set of stage events (not in the timed region: "
                                 "they cost ~50 us per step)" % n_stage}
    dense_bytes = sum(f.numel() * 4 for f in feats_h)
    row_bytes = sum(NS) * Cdim * 4
    if "zero_fill" in stage_ms:
        # the zero fill of the dense gradients + gradient rows: a library memset on a side stream, timed on that stream
        fill_bytes = dense_bytes + 4 * mod.last_state.sp.dF_n
        roofline["zero_fill_hbm"] = {"kernel": "cudaMemsetAsync (side stream, overlaps the sampling / gather stages)",
                                     "bytes": fill_bytes, "launch_ms": stage_ms["zero_fill"],
                                     "achieved_gbs": fill_bytes / (stage_ms["zero_fill"] * 1e-3) / 1e9,
                                     "peak_gbs": pk["hbm"]}
    if args.layout == "nchw":
        from mscs_b200 import _ops as _o
        if _o._DENSE_ONE_PASS:
            # default path: k_dx_rows (gradient rows + unit rows read, dx rows written) + k_dense_stream (slot maps and
            # dx rows read, EVERY byte of the dense gradients written once; no memset anywhere)
            sc_bytes = 3 * row_bytes + 4 * sum(f.shape[0] * f.shape[2] * f.shape[3] for f in feats_h) + row_bytes \
                + dense_bytes
            roofline["scatter_hbm"] = {"kernel": "k_dx_rows + k_dense_stream (one-pass dense-gradient writer)",
                                       "bytes": sc_bytes, "dense_gradient_bytes_written": dense_bytes,
                                       "achieved_gbs": sc_bytes / (stage_ms["scatter"] * 1e-3) / 1e9,
                                       "peak_gbs": pk["hbm"], "launch_ms": stage_ms["scatter"],
                                       "note": "pure-write stream: the measured memset rate on this part is ~4.7 TB/s; "
                                               "peak_gbs is the copy (read + write) figure of MEASURED_PEAKS.json"}
        else:
            # MSCS_DENSE=0: the scatter kernel's OWN algorithmic bytes: gradient rows + unit rows read, slot maps read,
            # one 32-byte sector written per sampled pixel and channel (the dense zero fill is the separate entry above)
            sc_bytes = 2 * row_bytes + 4 * sum(f.shape[0] * f.shape[2] * f.shape[3] for f in feats_h) \
                + sum(NS) * Cdim * 32
            roofline["scatter_hbm"] = {"kernel": "k_scatter_sectors_batch", "bytes": sc_bytes,
                                       "achieved_gbs": sc_bytes / (stage_ms["scatter"] * 1e-3) / 1e9,
                                       "peak_gbs": pk["hbm"], "launch_ms": stage_ms["scatter"]}
        # gather: useful bytes (N*C*4 read + rows written) and the sector traffic NCHW forces (one 32 B sector per value)
        roofline["gather_hbm"] = {"kernel": "k_gather_sectors_batch", "bytes": row_bytes + sum(NS) * (Cdim * 6 + 4),
                                  "sector_bytes": sum(NS) * Cdim * 32 + sum(NS) * (Cdim * 6 + 4),
                                  "achieved_gbs": (sum(NS) * Cdim * 32 + sum(NS) * (Cdim * 6 + 4))
                                  / (stage_ms["gather"] * 1e-3) / 1e9,
                                  "peak_gbs": pk["hbm"], "launch_ms": stage_ms["gather"]}
    else:
        # row kernels: the stage times hold the row traffic only (the zero fill of the dense gradients runs on the side
        # stream under the other stages); latency-bound at this size, reported for completeness
        roofline["gather_hbm"] = {"kernel": "k_gather_rows_nhwc", "bytes": row_bytes + sum(NS) * (Cdim * 6 + 4),
                                  "achieved_gbs": (row_bytes + sum(NS) * (Cdim * 6 + 4)) / (stage_ms["gather"] * 1e-3) / 1e9,
                                  "peak_gbs": pk["hbm"], "launch_ms": stage_ms["gather"]}
        roofline["scatter_hbm"] = {"kernel": "k_scatter_rows_nhwc", "bytes": 3 * row_bytes,
                                   "achieved_gbs": 3 * row_bytes / (stage_ms["scatter"] * 1e-3) / 1e9,
                                   "peak_gbs": pk["hbm"], "launch_ms": stage_ms["scatter"]}

    # ---- the sharded (pooled cross-batch) configuration next to the replica numbers ---------------
    pooled_rec = None
    if not pooled and not args.no_pooled:
        del feats, labels
        torch.cuda.empty_cache()
        pooled_rec = measure_pooled(dev, rank, world, dist)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if pooled else "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": bench_config(args.workload, world, args.layout),
            "detail": {"anchors_per_scale": NS, "anchor_pairs_per_step": pairs, "loss": float(loss.detach())},
            "roofline": roofline, "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": n_e2e,
                    "pipeline": "the copy of step i+1's inputs (copy stream) overlaps step i's kernels; every step "
                                "copies its own inputs and reads its loss back; the dense feature gradients (the "
                                "backward's result, 535 MB at cfg2) STAY on the device, where the projector's backward "
                                "consumes them in training",
                    "serial_ms_per_step": e2e_serial_ms},
            "gpu_launches": _ops.LAUNCHES_PER_STEP(len(feats_h), cfg["single_scale"]) * args.steps}
    if pooled_rec is not None:
        line["pooled"] = pooled_rec
    if not args.no_cpu_baseline and world == 1:
        # bounded sample (~20 s of CPU work): the reference's own files on the first 3 images, 1 warm-up + 2 timed steps
        cb = cpu_sample(args.workload, 2, 1, budget_s=60.0, images=min(CPU_SAMPLE_IMAGES, cfg["n"]))
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
