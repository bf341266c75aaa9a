"""Pooled mode at cfg-5 (64 images over the ranks, one process per GPU) with bf16 maps read natively, against the same
maps run through an fp32 copy (what the pooled mode did before it read half maps) and against fp32 maps.  Arms
alternated over several rounds in the same call; device events around forward + backward on every rank.

    fp32         fp32 maps
    bf16_native  bf16 maps handed to the loss; gradients come back in bf16
    bf16_upcast  bf16 maps, x.float() outside the loss, fp32 loss, .to(bf16) of the gradients

Per rank and arm: ms per step (median over rounds, and every round) and the peak increase of max_memory_allocated over
one step.  Rank 0 writes <out>/pooled_io_<world>gpu.json with every rank's card name, power limit and max SM clock read
in the same call.

    torchrun --nproc-per-node N tools/pooled_io_bench.py --out DIR [--layout nchw] [--rounds 5] [--steps 10] [--warmup 3]
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
    ap.add_argument("--out", required=True, help="directory that receives pooled_io_<world>gpu.json (rank 0)")
    ap.add_argument("--layout", choices=["nchw", "channels_last"], default="nchw")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    import mscs_b200
    from mscs_b200 import synth
    assert torch.cuda.is_available(), "pooled_io_bench.py measures on GPUs; there is no CPU fallback"
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    bf16 = torch.bfloat16
    fmt = torch.channels_last if args.layout == "channels_last" else torch.contiguous_format

    cfg = synth.CONFIGS["cfg5"]
    labels_h, feats_h = synth.make_inputs("cfg5")
    nl = labels_h.shape[0] // world
    labels = labels_h[rank * nl:(rank + 1) * nl].to(dev)
    f32 = [f[rank * nl:(rank + 1) * nl].to(dev).contiguous(memory_format=fmt).requires_grad_(True) for f in feats_h]
    fbf = [f.detach().to(bf16).contiguous(memory_format=fmt).requires_grad_(True) for f in f32]
    del labels_h, feats_h
    mods = {k: mscs_b200.DenseContrastiveLossV2_ms(dict(cfg["loss"]), comm=mscs_b200.TorchDistComm())
            for k in ("fp32", "bf16_native", "bf16_upcast")}
    torch.manual_seed(0)            # the reference sampler: every rank's generator in the same state

    def fp32():
        return torch.autograd.grad(mods["fp32"](labels, f32), f32)

    def native():
        return torch.autograd.grad(mods["bf16_native"](labels, fbf), fbf)

    def upcast():
        x = [f.detach().float().contiguous(memory_format=fmt).requires_grad_(True) for f in fbf]
        return [g.to(bf16) for g in torch.autograd.grad(mods["bf16_upcast"](labels, x), x)]

    arms = {"fp32": fp32, "bf16_native": native, "bf16_upcast": upcast}
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
        grads = fn()
        torch.cuda.synchronize()
        return (torch.cuda.max_memory_allocated(dev) - base) / 1e6, str(grads[0].dtype)

    mine = {"rank": rank, "gpu": gpu_facts(local), "arms": {}}
    for k, fn in arms.items():
        peak, dt = peak_mb(fn)
        mine["arms"][k] = {"ms_per_step_median": statistics.median(rounds[k]), "ms_per_step_rounds": rounds[k],
                           "peak_alloc_increase_mb": peak, "grad_dtype": dt}
    every = [None] * world
    dist.all_gather_object(every, mine)
    if rank == 0:
        result = {"config": "cfg5", "world": world, "layout": args.layout, "images_per_rank": nl,
                  "torch": torch.__version__, "lib": mscs_b200.load().mscs_version().decode(), "rounds": args.rounds,
                  "steps_per_round": args.steps, "warmup": args.warmup, "ranks": every}
        os.makedirs(args.out, exist_ok=True)
        path = os.path.join(args.out, f"pooled_io_{world}gpu.json")
        with open(path, "w") as fh:
            json.dump(result, fh, indent=1)
        for r in every:
            print(json.dumps({"rank": r["rank"], "gpu": r["gpu"].splitlines()[-1],
                              **{k: [round(v["ms_per_step_median"], 4), round(v["peak_alloc_increase_mb"], 1)]
                                 for k, v in r["arms"].items()}}))
        print("wrote", path)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
