"""2+ GPU check of the pooled mode under torchrun: every rank compares its pooled loss / gradients
with the single-process loss of the concatenated batch computed locally.

  torchrun --nproc-per-node N tools/pooled_check.py [cfg5] [--dtype bf16] [--layout channels_last] [--sampler philox]
                                                   [--tail]

--dtype / --layout / --sampler: element type and memory format of the feature maps (both runs get the same maps) and
the sampler.  cfg5: also BASELINE config 5 (fp32 NCHW maps, reference sampler) against the fp64-oracle fixture.
--tail: the projector tail (ProjectorTailContrastive_ms, c_prev 64 -> d 64, the same weights on every rank) instead of
the drop-in class on the maps; the sum over the ranks of the weight and bias gradients is compared with the
single-process ones (within 1e-3 of their maximum)."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
import mscs_b200
from mscs_b200 import synth

ap = argparse.ArgumentParser()
ap.add_argument("mode", nargs="?", choices=["cfg5"])
ap.add_argument("--dtype", choices=["fp32", "bf16", "fp16"], default="fp32")
ap.add_argument("--layout", choices=["nchw", "channels_last"], default="nchw")
ap.add_argument("--sampler", choices=["reference", "philox"], default="reference")
ap.add_argument("--tail", action="store_true")
args = ap.parse_args()
dtype = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[args.dtype]
fmt = torch.channels_last if args.layout == "channels_last" else torch.contiguous_format

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
cfg = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
           cross_scale_contrast=True, w_high_low=0.5, w_high_mid=0.25, min_views_per_class=5,
           max_views_per_class=50, max_features_total=3000, sampler=args.sampler, sampler_seed=11)
n = 2 * world
labels = synth.synth_labels(n, 128, 256, 19, 7, 16, 0.05, 21)
feats = synth.synth_features(n, 64, 128, 256, [4, 8, 16], 22)


def make(comm=None):
    if not args.tail:
        return mscs_b200.DenseContrastiveLossV2_ms(dict(cfg), comm=comm)
    torch.manual_seed(3)            # the same tails on every rank and in the single process
    return mscs_b200.ProjectorTailContrastive_ms(dict(cfg), 64, 64, comm=comm).to(dev)


full = make()
fg = [f.to(dev).to(dtype).contiguous(memory_format=fmt).requires_grad_(True) for f in feats]
torch.manual_seed(5)
loss_full = full(labels.to(dev), fg)
loss_full.backward()
nl = n // world
mod = make(mscs_b200.TorchDistComm())
fl = [f[rank * nl:(rank + 1) * nl].to(dev).to(dtype).contiguous(memory_format=fmt).requires_grad_(True) for f in feats]
torch.manual_seed(5)
loss = mod(labels[rank * nl:(rank + 1) * nl].to(dev), fl)
loss.backward()
torch.cuda.synchronize()
ok = abs(float(loss) - float(loss_full)) < 2e-5 * abs(float(loss_full))
for s in range(len(fl)):
    ok = ok and fl[s].grad.dtype == dtype and fl[s].grad.stride() == fl[s].stride()
    g, w = (x.float().cpu().numpy().ravel().astype(np.float64) for x in (fl[s].grad, fg[s].grad[rank * nl:(rank + 1) * nl]))
    cos = float(g @ w / np.sqrt((g @ g) * (w @ w)))
    ok = ok and cos > 0.99999 and np.array_equal(g != 0, w != 0)
    print(f"rank {rank} scale {s}: cosine {cos:.8f} max-abs {np.abs(g - w).max():.3e}", flush=True)
if args.tail:
    for name, mine, ref in [(f"{k}{s}", getattr(t, k).grad.clone(), getattr(u, k).grad)
                            for k in ("weight", "bias") for s, (t, u) in enumerate(zip(mod.tails, full.tails))]:
        dist.all_reduce(mine)           # the ranks' contributions
        err = float((mine - ref).abs().max()) / float(ref.abs().max())
        ok = ok and err <= 1e-3
        print(f"rank {rank} tail {name}: sum over ranks vs single process, max-abs / max {err:.3e}", flush=True)
print(f"rank {rank} ({'tail, ' if args.tail else ''}{args.dtype}, {args.layout}, sampler {args.sampler}): pooled loss {float(loss):.6f} single-process "
      f"{float(loss_full):.6f} -> {'OK' if ok else 'MISMATCH'}", flush=True)

if args.mode == "cfg5":
    # BASELINE config 5 over real ranks against the fp64-oracle fixture (tests/golden/cfg5.npz): loss, term losses and
    # the recorded gradient rows of the pixels this rank owns
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    meta = json.load(open(os.path.join(root, "tests", "golden", "golden.json")))["cfg5"]
    z = np.load(os.path.join(root, "tests", "golden", "cfg5.npz"))
    labels5, feats5 = synth.make_inputs("cfg5")
    nl5 = labels5.shape[0] // world
    mod5 = mscs_b200.DenseContrastiveLossV2_ms(dict(meta["loss_cfg"]), comm=mscs_b200.TorchDistComm())
    f5 = [f[rank * nl5:(rank + 1) * nl5].to(dev).requires_grad_(True) for f in feats5]
    torch.manual_seed(0)
    loss5 = mod5(labels5[rank * nl5:(rank + 1) * nl5].to(dev), f5)
    loss5.backward()
    torch.cuda.synchronize()
    rel = abs(float(loss5) - meta["total"]) / abs(meta["total"])
    ok5 = rel < 1e-3
    for a, b in zip([float(x) for x in mod5.ms_losses] + [float(x) for x in mod5.cs_losses], meta["ms"] + meta["cs"]):
        ok5 = ok5 and abs(a - b) < 1e-3 * abs(b)
    for s in range(len(f5)):
        idx, pairs, ids = z[f"idx{s}"], z[f"pairs{s}"], z[f"grad_row_ids{s}"]
        V = idx.shape[1]
        got, want = [], []
        for j, i in enumerate(ids):
            k, v = i // V, i % V
            b = int(pairs[k, 0])
            if b // nl5 != rank:
                continue
            g = f5[s].grad[b % nl5]
            got.append(g.reshape(g.shape[0], -1)[:, int(idx[k, v])].cpu().numpy())
            want.append(z[f"grad_rows{s}"][j])
        if got:
            g_, w_ = np.concatenate(got).astype(np.float64), np.concatenate(want).astype(np.float64)
            cos = float(g_ @ w_ / np.sqrt((g_ @ g_) * (w_ @ w_)))
            ok5 = ok5 and cos >= 0.999
            print(f"rank {rank} cfg5 scale {s}: {len(got)} fixture rows owned, cosine {cos:.7f} max-abs {np.abs(g_ - w_).max():.3e}", flush=True)
    print(f"rank {rank}: cfg5 pooled loss {float(loss5):.6f} fp64 oracle {meta['total']:.6f} rel {rel:.2e} -> {'OK' if ok5 else 'MISMATCH'}", flush=True)
    ok = ok and ok5
dist.destroy_process_group()
sys.exit(0 if ok else 1)
