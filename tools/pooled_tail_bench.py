"""Projector tail in the pooled mode at cfg-5 (64 images over the ranks, one process per GPU), c_prev = d = 256, fp32
NCHW maps z in front of the projector's last 1x1 convolution.  Two arms in the same process, alternated over rounds:

    dense  nn.Conv2d(c_prev, d, 1) on every pixel of every local image, then the pooled drop-in
           DenseContrastiveLossV2_ms(config, comm) on the projected maps
    tail   ProjectorTailContrastive_ms(config, c_prev, d, comm): only this rank's sampled rows are projected

Each step is forward + backward to z and to the convolution's weight and bias.  Per arm: ms per step from device events
(the median over rounds of every rank's time, and its maximum over the ranks), and each rank's peak increase of
max_memory_allocated over one step.  For the tail also the gap between the end of the raw gather and the start of the
GEMM (the forward's one host wait for the plan records and local row counts), from device events, median over steps.
Rank 0 writes <out>/pooled_tail_<world>gpu.json with every rank's card name, power limit and max SM clock read in the
same call.

    torchrun --nproc-per-node N tools/pooled_tail_bench.py --out DIR [--rounds 5] [--steps 10] [--warmup 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_facts(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory that receives pooled_tail_<world>gpu.json (rank 0)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    import torch.nn as nn
    import mscs_b200
    from mscs_b200 import _ops, synth
    assert torch.cuda.is_available(), "pooled_tail_bench.py measures on GPUs; there is no CPU fallback"
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)

    cfg = synth.CONFIGS["cfg5"]
    labels_h, feats_h = synth.make_inputs("cfg5")
    c_prev = d = feats_h[0].shape[1]
    assert c_prev == 256
    nl = labels_h.shape[0] // world
    labels = labels_h[rank * nl:(rank + 1) * nl].to(dev)
    zs = [f[rank * nl:(rank + 1) * nl].to(dev).contiguous().requires_grad_(True) for f in feats_h]
    del labels_h, feats_h
    torch.manual_seed(3)
    tail = mscs_b200.ProjectorTailContrastive_ms(dict(cfg["loss"]), c_prev, d, comm=mscs_b200.TorchDistComm()).to(dev)
    convs = nn.ModuleList([nn.Conv2d(c_prev, d, 1) for _ in zs]).to(dev)
    convs.load_state_dict(tail.tails.state_dict())
    drop = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg["loss"]), comm=mscs_b200.TorchDistComm())
    torch.manual_seed(0)            # the reference sampler: every rank's generator in the same state

    def dense():
        params = [p for c in convs for p in (c.weight, c.bias)]
        return torch.autograd.grad(drop(labels, [c(z) for c, z in zip(convs, zs)]), zs + params)

    def projected():
        params = [p for t in tail.tails for p in (t.weight, t.bias)]
        return torch.autograd.grad(tail(labels, zs), zs + params)

    arms = {"dense": dense, "tail": projected}
    for fn in arms.values():
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    rounds = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            e1.synchronize()
            rounds[k].append(e0.elapsed_time(e1) / args.steps)

    def peak_mb(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        fn()
        torch.cuda.synchronize()
        return (torch.cuda.max_memory_allocated(dev) - base) / 1e6

    mine = {"rank": rank, "gpu": gpu_facts(local), "arms": {}}
    for k, fn in arms.items():
        mine["arms"][k] = {"ms_per_step_median": statistics.median(rounds[k]), "ms_per_step_rounds": rounds[k],
                           "peak_alloc_increase_mb": peak_mb(fn)}
    # the host-wait gap of the tail's forward, in a pass of its own (the events are recorded only when asked for)
    _ops.TIMING = {}
    for _ in range(args.steps):
        projected()
    torch.cuda.synchronize()
    gaps = [a.elapsed_time(b) for a, b in _ops.TIMING["tail_wait_gap"]]
    _ops.TIMING = None
    mine["tail_wait_gap_ms"] = {"median": statistics.median(gaps), "max": max(gaps), "steps": len(gaps)}
    every = [None] * world
    dist.all_gather_object(every, mine)
    if rank == 0:
        summary = {k: {"ms_per_step_max_over_ranks": max(r["arms"][k]["ms_per_step_median"] for r in every),
                       "peak_alloc_increase_mb_max_over_ranks": max(r["arms"][k]["peak_alloc_increase_mb"]
                                                                    for r in every)} for k in arms}
        summary["tail_wait_gap_ms_median_max_over_ranks"] = max(r["tail_wait_gap_ms"]["median"] for r in every)
        result = {"config": "cfg5", "world": world, "images_per_rank": nl, "c_prev": c_prev, "d": d,
                  "maps": "fp32 NCHW", "torch": torch.__version__, "lib": mscs_b200.load().mscs_version().decode(),
                  "rounds": args.rounds, "steps_per_round": args.steps, "warmup": args.warmup, "summary": summary,
                  "ranks": every}
        os.makedirs(args.out, exist_ok=True)
        path = os.path.join(args.out, f"pooled_tail_{world}gpu.json")
        with open(path, "w") as fh:
            json.dump(result, fh, indent=1)
        print(json.dumps({"world": world, "gpu": every[0]["gpu"].splitlines()[-1], **summary}))
        print("wrote", path)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
