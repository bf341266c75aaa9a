"""The projector's last 1x1 convolution + the loss, forward + backward, at the cfg-2 shape (12 images, c_prev = d = 256,
512x1024, strides 4/8/16/32): the dense evaluation against ProjectorTailContrastive_ms.  One process on one GPU, arms
alternated over several rounds in the same call (the scheme of tools/graph_bench.py).

  dense_fp32           nn.Conv2d on every pixel + DenseContrastiveLossV2_ms, fp32 maps
  dense_bf16_autocast  the same under torch.autocast(bfloat16): the convolution emits bf16 maps, read natively
  tail_fp32            ProjectorTailContrastive_ms, eager, fp32 maps z
  tail_bf16            the same on bf16 maps z
  tail_graph_philox    g.replay() of a tail step captured with sampler='philox' (fp32 maps)
  parent_tail_fp32     (--parent DIR) the tail module of another checkout, loaded from DIR, fp32 maps

Every arm computes the gradients w.r.t. the maps z, the weights and the biases (torch.autograd.grad).  Per arm: ms per
step from device events around `--steps` back-to-back steps (median over rounds, and every round), and the peak
allocation of one step above what was allocated before it.  Writes <out>/projector_tail.json with the card name, power
limit and max SM clock read in the same call.

    python tools/projector_tail_bench.py --out DIR [--parent DIR] [--rounds 5] [--steps 20] [--warmup 5]
"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "eccv2022-multi-scale-and-cross-scale-contrastive-segmentation_b200"


def gpu_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def load_other(root, name):
    """The package of another checkout (its own libmscs.so) under the module name `name`."""
    d = os.path.join(os.path.abspath(root), PKG)
    spec = importlib.util.spec_from_file_location(name, os.path.join(d, "__init__.py"), submodule_search_locations=[d])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory that receives projector_tail.json")
    ap.add_argument("--parent", default=None, help="another checkout (built) whose tail module runs as one more arm")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()

    import torch
    import mscs_b200
    from mscs_b200 import synth
    assert torch.cuda.is_available(), "projector_tail_bench.py measures on a GPU; there is no CPU fallback"
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_facts(), "torch": torch.__version__, "lib": mscs_b200.load().mscs_version().decode(),
              "shape": "cfg2: 12 x 256 x 512/s x 1024/s, s = 4, 8, 16, 32; d = 256", "rounds": args.rounds,
              "steps_per_round": args.steps, "warmup": args.warmup}
    cfg = dict(synth.CONFIGS["cfg2"]["loss"])
    labels = synth.synth_labels(12, 512, 1024, 19, 19, 32, 0.05, 0).to(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    z32 = [torch.randn(12, 256, 512 // s, 1024 // s, device=dev, generator=g).requires_grad_(True) for s in (4, 8, 16, 32)]
    z16 = [z.detach().to(torch.bfloat16).requires_grad_(True) for z in z32]
    torch.manual_seed(0)
    tail = mscs_b200.ProjectorTailContrastive_ms(cfg, 256, 256).to(dev)
    params = [t.weight for t in tail.tails] + [t.bias for t in tail.tails]
    drop = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg))

    def dense():
        torch.autograd.grad(drop(labels, [t(z) for t, z in zip(tail.tails, z32)]), z32 + params)

    def dense_ac():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = drop(labels, [t(z) for t, z in zip(tail.tails, z32)])
        torch.autograd.grad(loss, z32 + params)

    arms = {"dense_fp32": dense, "dense_bf16_autocast": dense_ac,
            "tail_fp32": lambda: torch.autograd.grad(tail(labels, z32), z32 + params),
            "tail_bf16": lambda: torch.autograd.grad(tail(labels, z16), z16 + params)}

    ph = mscs_b200.ProjectorTailContrastive_ms(dict(cfg, sampler="philox", sampler_seed=1), 256, 256).to(dev)
    ph.load_state_dict(tail.state_dict())
    ph_params = [t.weight for t in ph.tails] + [t.bias for t in ph.tails]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            torch.autograd.grad(ph(labels, z32), z32 + ph_params)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        torch.autograd.grad(ph(labels, z32), z32 + ph_params)
    arms["tail_graph_philox"] = graph.replay

    if args.parent:
        other = load_other(args.parent, "mscs_parent")
        result["parent_lib"] = other.load().mscs_version().decode()
        ptail = other.ProjectorTailContrastive_ms(cfg, 256, 256).to(dev)
        ptail.load_state_dict(tail.state_dict())
        pparams = [t.weight for t in ptail.tails] + [t.bias for t in ptail.tails]
        arms["parent_tail_fp32"] = lambda: torch.autograd.grad(ptail(labels, z32), z32 + pparams)

    for fn in arms.values():
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    peak = {}
    for k, fn in arms.items():      # one step each: allocation above the state before it
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        peak[k] = (torch.cuda.max_memory_allocated() - base) / 2 ** 20
    dev_ms = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            e1.synchronize()
            dev_ms[k].append(e0.elapsed_time(e1) / args.steps)
    result["arms"] = {k: {"ms_per_step_median": statistics.median(v), "ms_per_step_rounds": v,
                          "spread_ms": max(v) - min(v), "peak_alloc_MiB": peak[k]} for k, v in dev_ms.items()}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "projector_tail.json")
    with open(path, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"gpu": result["gpu"], **{k: [round(v["ms_per_step_median"], 4), round(v["peak_alloc_MiB"], 1)]
                                               for k, v in result["arms"].items()}}))
    print("wrote", path)


if __name__ == "__main__":
    main()
