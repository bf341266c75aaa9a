"""Per-stage device times of cfg2 steps (run on a GPU)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import mscs_b200
from mscs_b200 import synth, _ops
dev = torch.device("cuda:0")
name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
cfg = synth.CONFIGS[name]
labels, feats = synth.make_inputs(name)
cls = mscs_b200.DenseContrastiveLossV2 if cfg["single_scale"] else mscs_b200.DenseContrastiveLossV2_ms
mod = cls(dict(cfg["loss"]))
labels = labels.to(dev); fg = [f.to(dev).requires_grad_(True) for f in feats]
torch.manual_seed(0)
def step():
    for f in fg: f.grad = None
    mod(labels, fg[0] if cfg["single_scale"] else fg).backward()
for _ in range(3): step()
_ops.TIMING = {}
for _ in range(10): step()
torch.cuda.synchronize()
import time
_ops.TIMING = None
_ops.HOST_WAIT = []
_ops.HOST_SEG = {}
_orig_fwd, _orig_bwd = _ops.run_forward, _ops.run_backward
def _tf(*a, **k):
    t = time.perf_counter(); r = _orig_fwd(*a, **k); _ops.HOST_SEG["run_forward total"] = _ops.HOST_SEG.get("run_forward total", 0.0) + time.perf_counter() - t; return r
def _tb(*a, **k):
    t = time.perf_counter(); r = _orig_bwd(*a, **k); _ops.HOST_SEG["run_backward total"] = _ops.HOST_SEG.get("run_backward total", 0.0) + time.perf_counter() - t; return r
_ops.run_forward, _ops.run_backward = _tf, _tb
t0 = time.perf_counter()
for _ in range(50): step()
t_enq = time.perf_counter() - t0
_ops.run_forward, _ops.run_backward = _orig_fwd, _orig_bwd
print({k: round(v / 50 * 1e6) for k, v in _ops.HOST_SEG.items()}, "us/step")
_ops.HOST_SEG = None
torch.cuda.synchronize()
t_all = time.perf_counter() - t0
print(f"wall/step {t_all/50*1e3:.3f} ms; host blocked in the plan fetch {sum(_ops.HOST_WAIT)/50*1e3:.3f} ms/step -> host busy {(t_enq-sum(_ops.HOST_WAIT))/50*1e3:.3f} ms/step")
_ops.TIMING = {}
for _ in range(30): step()
torch.cuda.synchronize()
print({k: round(sum(a.elapsed_time(b) for a, b in v) / len(v), 4) for k, v in _ops.TIMING.items()})

if os.environ.get("MSCS_FWD_TIMELINE"):
    import ctypes, numpy as np
    from mscs_b200 import _lib
    buf = np.zeros(8, np.float32)
    acc = np.zeros(8)
    for _ in range(10):
        step()
        n = _lib.load().mscs_debug_fwd_timeline(buf.ctypes.data, 8)
        acc[:n] += buf[:n]
    print("forward timeline (us): row_ranges, work0, sweep0, work1, sweep1, finalise =", [round(float(x) * 100, 1) for x in acc[:n]])
