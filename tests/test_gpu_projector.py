"""GPU: the projector tail evaluated on the sampled rows only (SURVEY.md 8f item 1, mscs_b200/projector.py) against the
DENSE evaluation it replaces -- ``nn.Conv2d(c_prev, d, 1)`` on every pixel (the last layer of the reference's
projector, models/Projector.py:69) followed by the fp64 oracle of ``DenseContrastiveLossV2_ms`` and by this repository's
drop-in class.  Same labels, same generator state: the sampled
pixels are identical, so loss and the gradients w.r.t. the pre-projection features, the weights and the biases must
agree within the north_star tolerances (loss 1e-3 relative, gradient cosine >= 0.999)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm()))


def _case(dev, n, c_prev, d, H, W, strides, cfg, seed):
    from mscs_b200 import synth
    from mscs_b200.projector import ProjectorTailContrastive_ms
    labels = synth.synth_labels(n, H, W, 19, 7, 16, 0.05, seed).to(dev)
    g = torch.Generator().manual_seed(seed + 1)
    zs = [torch.randn(n, c_prev, H // s, W // s, generator=g).to(dev) for s in strides]
    torch.manual_seed(seed + 2)
    mod = ProjectorTailContrastive_ms(cfg, c_prev, d).to(dev)
    return labels, zs, mod


def _run_sparse(mod, labels, zs, rng):
    zg = [z.clone().requires_grad_(True) for z in zs]
    mod.zero_grad()
    torch.set_rng_state(rng)
    loss = mod(labels, zg)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), [z.grad for z in zg], [t.weight.grad.clone() for t in mod.tails], \
        [t.bias.grad.clone() for t in mod.tails]


def _run_dense(loss_mod, mod, labels, zs, rng):
    zg = [z.clone().requires_grad_(True) for z in zs]
    mod.zero_grad()
    torch.set_rng_state(rng)
    loss = loss_mod(labels, [t(z) for t, z in zip(mod.tails, zg)])
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), [z.grad for z in zg], [t.weight.grad.clone() for t in mod.tails], \
        [t.bias.grad.clone() for t in mod.tails]


CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
           cross_scale_contrast=True, w_high_low=0.5, w_high_mid=0.25, min_views_per_class=5,
           max_views_per_class=40, max_features_total=1200)


def test_projector_tail_vs_dense_fp64_oracle(dev):
    """The dense evaluation with the fp64 oracle as the loss: ``nn.Conv2d`` on every pixel, oracle loss and gradient
    w.r.t. the projected maps, autograd back through the convolutions."""
    from oracle import loss_fp64
    from oracle.config import oracle_cfg
    from oracle.mt19937 import MT19937
    labels, zs, mod = _case(dev, 3, 48, 64, 128, 256, [4, 8, 16], CFG, 31)
    torch.manual_seed(9)
    rng = torch.get_rng_state()
    l_s, gz_s, gw_s, gb_s = _run_sparse(mod, labels, zs, rng)
    rng_after = MT19937.from_torch_state(torch.get_rng_state().numpy().tobytes())
    zg = [z.clone().requires_grad_(True) for z in zs]
    mod.zero_grad()
    ys = [t(z) for t, z in zip(mod.tails, zg)]
    gen = MT19937.from_torch_state(rng.numpy().tobytes())
    res = loss_fp64.ms_cs_loss(labels.cpu().numpy(), [y.detach().cpu().double().numpy() for y in ys],
                               oracle_cfg(CFG, 20), gen)
    assert gen.pos == rng_after.pos and np.array_equal(gen.mt, rng_after.mt)
    torch.autograd.backward(ys, [torch.from_numpy(g).to(dev, torch.float32) for g in res["grads"]])
    torch.cuda.synchronize()
    l_r, gz_r = res["total"], [z.grad for z in zg]
    gw_r, gb_r = [t.weight.grad.clone() for t in mod.tails], [t.bias.grad.clone() for t in mod.tails]
    rel = abs(float(l_s) - l_r) / abs(l_r)
    print(f"projector tail: loss {float(l_s):.6f} dense fp64 oracle {l_r:.6f} rel {rel:.2e}")
    assert rel < 1e-3
    for s in range(len(zs)):
        assert torch.equal((gz_s[s] != 0).any(dim=1), (gz_r[s] != 0).any(dim=1)), "different pixels carry a gradient"
        cz, cw, cb = _cos(gz_s[s], gz_r[s]), _cos(gw_s[s], gw_r[s]), _cos(gb_s[s], gb_r[s])
        print(f"  scale {s}: cosine dz {cz:.7f} dW {cw:.7f} db {cb:.7f}; max-abs dz "
              f"{float((gz_s[s] - gz_r[s]).abs().max()):.3e} dW {float((gw_s[s] - gw_r[s]).abs().max()):.3e}")
        assert cz >= 0.999 and cw >= 0.999 and cb >= 0.999
    assert [float(x) for x in mod.ms_losses] and len(mod.cs_losses) == 2


def test_projector_tail_vs_own_dense_path_cfg2_shape(dev):
    """HRNet-W48 Cityscapes shape (c_prev = d = 256, 12 images): against this repository's drop-in class on the dense
    projector output (same kernels after the projection: the two must agree to fp32 rounding of the GEMM)."""
    import time
    import mscs_b200
    from mscs_b200 import synth
    cfg = dict(synth.CONFIGS["cfg2"]["loss"])
    labels, zs, mod = _case(dev, 12, 256, 256, 512, 1024, [4, 8, 16, 32], cfg, 41)
    torch.manual_seed(3)
    rng = torch.get_rng_state()
    l_s, gz_s, gw_s, gb_s = _run_sparse(mod, labels, zs, rng)
    dense = mscs_b200.DenseContrastiveLossV2_ms(cfg)
    l_d, gz_d, gw_d, gb_d = _run_dense(dense, mod, labels, zs, rng)
    assert abs(float(l_s) - float(l_d)) < 1e-4 * abs(float(l_d)), (float(l_s), float(l_d))
    for s in range(len(zs)):
        assert _cos(gz_s[s], gz_d[s]) > 0.9999 and _cos(gw_s[s], gw_d[s]) > 0.9999 and _cos(gb_s[s], gb_d[s]) > 0.9999
        assert torch.equal((gz_s[s] != 0).any(dim=1), (gz_d[s] != 0).any(dim=1))
    # timing of the two evaluations (events, 5 steps each after 2 warm-up): projection + loss, forward + backward
    def timed(fn):
        for _ in range(2):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 5
    t_sparse = timed(lambda: _run_sparse(mod, labels, zs, rng))
    t_dense = timed(lambda: _run_dense(dense, mod, labels, zs, rng))
    print(f"cfg2 shape, projection tail + loss, fwd+bwd: sampled rows only {t_sparse:.3f} ms, dense conv1x1 + drop-in loss "
          f"{t_dense:.3f} ms (includes the clone of the inputs in both)")
