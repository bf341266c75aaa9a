"""bf16 inputs read natively by the kernels against the same inputs run through an fp32 copy (what the library did before
it read half maps / logits), and against the fp32 headline path.  One process on one GPU, arms alternated over several
rounds in the same call; device events around forward + backward.

  contrastive (cfg-2, NCHW and channels-last):
    fp32         fp32 maps (bench.py's workload)
    bf16_native  bf16 maps handed to the loss; gradients come back in bf16
    bf16_upcast  bf16 maps, f.float() outside the loss, fp32 loss, .to(bf16) of the gradients
  cross entropy (CrossEntropyLabelPass, 12 x 19 x 512 x 1024, label pass made beforehand):
    fp32, bf16_native, bf16_upcast (logits.float(), fp32 CE, .to(bf16) of dlogits)

Per arm: ms per step (median over rounds, and every round), the gather / scatter stage times through _ops.TIMING (the
hooks bench.py uses; a separate pass, the events cost step time), and the peak increase of max_memory_allocated over
one step.  Writes <out>/half_io.json with the card name, power limit and max SM clock read in the same call.

    python tools/half_io_bench.py --out DIR [--rounds 5] [--steps 20] [--warmup 10]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory that receives half_io.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()

    import torch
    import mscs_b200
    from mscs_b200 import _ops, synth
    assert torch.cuda.is_available(), "half_io_bench.py measures on a GPU; there is no CPU fallback"
    dev = torch.device("cuda:0")
    bf16 = torch.bfloat16
    result = {"gpu": gpu_facts(), "torch": torch.__version__, "lib": mscs_b200.load().mscs_version().decode(),
              "rounds": args.rounds, "steps_per_round": args.steps, "warmup": args.warmup}

    def timed_rounds(arms):
        """{arm: [ms per step of each round]}, arms alternated inside every round."""
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        out = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    fn()
                e1.record()
                e1.synchronize()
                out[k].append(e0.elapsed_time(e1) / args.steps)
        return out

    def peak_mb(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        fn()
        torch.cuda.synchronize()
        return (torch.cuda.max_memory_allocated(dev) - base) / 1e6

    def stages(fn, n=10):
        _ops.TIMING, _ops.TIMING_ALL = {}, True
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        st = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in _ops.TIMING.items()}
        _ops.TIMING = None
        return {k: st[k] for k in ("gather", "scatter") if k in st}

    def summary(rounds, extra):
        return {k: {"ms_per_step_median": statistics.median(v), "ms_per_step_rounds": v, **extra[k]}
                for k, v in rounds.items()}

    # ---- contrastive loss, cfg-2 -------------------------------------------------------------------------------
    cfg = synth.CONFIGS["cfg2"]
    labels_h, feats_h = synth.make_inputs("cfg2")
    labels = labels_h.to(dev)
    torch.manual_seed(0)
    result["contrastive"] = {}
    for layout in ("nchw", "channels_last"):
        fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
        f32 = [f.to(dev).contiguous(memory_format=fmt).requires_grad_(True) for f in feats_h]
        fbf = [f.detach().to(bf16).contiguous(memory_format=fmt).requires_grad_(True) for f in f32]
        mods = {k: mscs_b200.DenseContrastiveLossV2_ms(dict(cfg["loss"])) for k in ("fp32", "bf16_native", "bf16_upcast")}

        def fp32():
            return torch.autograd.grad(mods["fp32"](labels, f32), f32)

        def native():
            return torch.autograd.grad(mods["bf16_native"](labels, fbf), fbf)

        def upcast():
            x = [f.detach().float().contiguous(memory_format=fmt).requires_grad_(True) for f in fbf]
            return [g.to(bf16) for g in torch.autograd.grad(mods["bf16_upcast"](labels, x), x)]

        arms = {"fp32": fp32, "bf16_native": native, "bf16_upcast": upcast}
        rounds = timed_rounds(arms)
        # gradient dtypes as a caller sees them (a sanity check of what was timed)
        dtypes = {k: str(fn()[0].dtype) for k, fn in arms.items()}
        extra = {k: {"stage_ms": stages(fn), "peak_alloc_increase_mb": peak_mb(fn), "grad_dtype": dtypes[k]}
                 for k, fn in arms.items()}
        result["contrastive"][layout] = summary(rounds, extra)
        del f32, fbf, mods, arms

    # ---- cross entropy, 12 x 19 x 512 x 1024 --------------------------------------------------------------------
    from mscs_b200.coloss import CITYSCAPES_CLASS_WEIGHTS
    g = torch.Generator().manual_seed(3)
    n, K, H, W = 12, 19, 512, 1024
    lab = synth.synth_labels(n, H, W, 19, 19, 32, 0.05, 0).to(dev)
    compact = mscs_b200.label_pass(lab, 20)
    x32 = (2.0 * torch.randn(n, K, H, W, generator=g)).to(dev).requires_grad_(True)
    xbf = x32.detach().to(bf16).requires_grad_(True)
    ce = mscs_b200.CrossEntropyLabelPass(20, 19, CITYSCAPES_CLASS_WEIGHTS).to(dev)

    def ce32():
        return torch.autograd.grad(ce(x32, compact), x32)

    def ce_native():
        return torch.autograd.grad(ce(xbf, compact), xbf)

    def ce_upcast():
        x = xbf.detach().float().requires_grad_(True)
        return [d.to(bf16) for d in torch.autograd.grad(ce(x, compact), x)]

    arms = {"fp32": ce32, "bf16_native": ce_native, "bf16_upcast": ce_upcast}
    rounds = timed_rounds(arms)
    extra = {k: {"peak_alloc_increase_mb": peak_mb(fn)} for k, fn in arms.items()}
    result["cross_entropy"] = {"shape": [n, K, H, W], **summary(rounds, extra)}

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "half_io.json")
    with open(path, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"gpu": result["gpu"],
                      **{f"{w}/{lay}/{k}": round(v["ms_per_step_median"], 4)
                         for w, block in (("contrastive", result["contrastive"]),)
                         for lay, arms_ in block.items() for k, v in arms_.items()},
                      **{f"ce/{k}": round(v["ms_per_step_median"], 4) for k, v in result["cross_entropy"].items()
                         if k != "shape"}}))
    print("wrote", path)


if __name__ == "__main__":
    main()
