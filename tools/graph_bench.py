"""The eager training step of the loss against the replay of the same step captured in a CUDA graph (cfg-2,
sampler='philox').  One process on one GPU, arms alternated over several rounds in the same call (the scheme of
tools/half_io_bench.py).

  eager   forward + backward (torch.autograd.grad) of DenseContrastiveLossV2_ms, called from Python every step
  graph   g.replay() of the same forward + backward captured once with torch.cuda.graph (the inputs stay in the static
          tensors; a training loop would copy its next batch into them first)

for NCHW fp32 and NCHW bf16 feature maps.  Per arm: ms per step from device events around `--steps` back-to-back steps
(median over rounds, and every round), and host ms per step: the wall time until the last step's calls have returned,
before the closing synchronisation.  Writes <out>/graph.json with the card name, power limit and max SM clock read in
the same call.

    python tools/graph_bench.py --out DIR [--rounds 7] [--steps 50] [--warmup 10]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory that receives graph.json")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()

    import torch
    import mscs_b200
    from mscs_b200 import synth
    assert torch.cuda.is_available(), "graph_bench.py measures on a GPU; there is no CPU fallback"
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_facts(), "torch": torch.__version__, "lib": mscs_b200.load().mscs_version().decode(),
              "config": "cfg2", "sampler": "philox", "rounds": args.rounds, "steps_per_round": args.steps,
              "warmup": args.warmup}
    cfg = dict(synth.CONFIGS["cfg2"]["loss"], sampler="philox", sampler_seed=1)
    labels_h, feats_h = synth.make_inputs("cfg2")
    labels = labels_h.to(dev)

    result["arms"] = {}
    for dname, dtype in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        maps = [f.to(dev, dtype).contiguous().requires_grad_(True) for f in feats_h]
        eager_mod = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg))
        graph_mod = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg))

        def eager():
            torch.autograd.grad(eager_mod(labels, maps), maps)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                torch.autograd.grad(graph_mod(labels, maps), maps)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            torch.autograd.grad(graph_mod(labels, maps), maps)

        arms = {"eager": eager, "graph": g.replay}
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        dev_ms = {k: [] for k in arms}
        host_ms = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                e0.record()
                for _ in range(args.steps):
                    fn()
                e1.record()
                t1 = time.perf_counter()
                e1.synchronize()
                dev_ms[k].append(e0.elapsed_time(e1) / args.steps)
                host_ms[k].append(1e3 * (t1 - t0) / args.steps)
        logged = graph_mod.fetch_logged()
        result["arms"][f"nchw_{dname}"] = {
            k: {"ms_per_step_median": statistics.median(dev_ms[k]), "ms_per_step_rounds": dev_ms[k],
                "spread_ms": max(dev_ms[k]) - min(dev_ms[k]),
                "host_ms_per_step_median": statistics.median(host_ms[k]), "host_ms_per_step_rounds": host_ms[k]}
            for k in arms}
        result["arms"][f"nchw_{dname}"]["graph_last_replay_total"] = logged["total"]
        result["arms"][f"nchw_{dname}"]["graph_call_index_end"] = int(graph_mod.graph_call_index)
        del g, maps, eager_mod, graph_mod, arms
        torch.cuda.synchronize()

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "graph.json")
    with open(path, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"gpu": result["gpu"],
                      **{f"{a}/{k}": [round(v["ms_per_step_median"], 4), round(v["host_ms_per_step_median"], 4)]
                         for a, block in result["arms"].items() for k, v in block.items() if isinstance(v, dict)}}))
    print("wrote", path)


if __name__ == "__main__":
    main()
