"""The kernels that move and normalise anchor rows -- the gathers + ``F.normalize(p=2, dim=1, eps=1e-12)`` (K2), the
normalisation backward + dense-gradient writers (the scatter half of K4) and their raw and pooled forms -- driven
directly through the C ABI on synthetic feature maps, pixel sets, slot maps and gradient rows, and compared row by row
with fp64 references.

Entry points (every dtype instance): ``mscs_gather_normalize``, ``mscs_gather_normalize_sectors_batch``,
``mscs_gather_rows_nhwc_batch``, ``mscs_gather_normalize_p2p``, ``mscs_gather_rows_p2p``, ``mscs_gather_raw_batch``,
``mscs_gather_raw_rows_batch``, ``mscs_scatter_grad``, ``mscs_scatter_sectors_batch``, ``mscs_scatter_dense_batch``,
``mscs_scatter_rows_nhwc_batch``, ``mscs_scatter_sectors_pull``, ``mscs_scatter_rows_pull``.

Error model (u = 2^-24, the unit roundoff of fp32; first order, with a (1 + 64 u) allowance for the second order).
Inputs are exact: a half map widens exactly to fp32, and the fp64 references start from that widening.

* Gather, per element: |f_c - u64_c| <= K_GATHER u |u64_c|, and |inv - inv64| <= K_INV u inv64, where
  u64 = x64 inv64 and inv64 = 1 / max(||x64||, 1e-12).  ``inv_norm_of`` sums squares of non-negative terms: per lane
  8 fmaf (the first term is rounded 8 times), then 5 warp_sum levels, so ss carries at most 13 roundings: 13 u
  relative.  sqrtf halves that and adds its own rounding, which is up to u like every correctly rounded operation:
  6.5 u + u = 7.5 u.  fmaxf is exact (on the clamp, 1e-12f is 1e-12 to within u).  The correctly rounded 1.f / x adds
  u: K_INV = 8.5.  The product v * inv adds u: K_GATHER = 9.5.
  An unfused evaluation has the same count: the product rounding of a term replaces the rounding fmaf would make.
* Scatter, the kernel alone (``dx_row`` on the fp32 f, inv and g it was given; fp64 reference
  dx64 = (g - f (f.g)) inv, or g inv where the kernel's inv >= 1e12f): per element
  |dx_c - dx64_c| <= K_DX u inv (|g_c| + |f_c| S),  S = sum_j |f_j g_j|.  The dot product has the shape of the sum of
  squares with signed terms: 13 u S.  It enters through f_c: 13 u |f_c| S.  f_c * dot rounds (u |f_c| S, unfused only),
  g - f dot rounds (u (|g_c| + |f_c| S)), the product by inv rounds (the same again): K_DX = 13 + 1 + 2 = 16 (the
  kernel's fused multiply-add saves one).  The bound is relative to inv (|g_c| + |f_c| S), not to |dx_c|, so rows with
  g parallel to f, whose dx cancels to almost 0, pass on the rounding of what cancelled.
* Scatter, the chain (gather, then scatter, against the autograd derivative of F.normalize at x, in fp64; below eps
  clamp_min passes no gradient through the norm, dx = g / eps): f = u64 (1 + 9.5 u), inv = inv64 (1 + 8.5 u), so f.g is
  off by 9.5 u S and f_c (f.g) by 19 u |u64_c| S; the inverse norm adds 8.5 u (|g_c| + |u64_c| S); dx_row adds K_DX:
  K_CHAIN = 19 + 8.5 + 16 = 43.5, relative to inv64 (|g_c| + |u64_c| S64).
* Exact (bit for bit, integer views): raw rows; every bf16 operand row is the round-to-nearest-even of the same
  kernel's fp32 unit row, with zeros in [C, C_pad) and in the padding rows [N, N_pad); the fp32 rows, inverse norms and
  bf16 rows of k_gather_normalize, k_gather_sectors_batch, k_gather_rows_nhwc and k_gather_rows_p2p are identical, and
  a half map gives the rows of its fp32 widening (k_gather_p2p sums in another order: the bound only, but identical bf16
  rows in every slab); every scatter gives the fp32 dx of mscs_scatter_grad, and a half gradient is that dx .to(dtype);
  the same call twice gives the same bytes.
* Write extents: every output is pre-filled with 0xFF bytes (a NaN in fp32, bf16 and fp16) inside 4 KiB guards of the
  same pattern; the guards must survive and each entry point writes exactly what include/mscs.h promises.  Inputs that
  must not be read hold NaN: the non-sampled pixels of the maps, dF columns [C, ldF), dF rows at or above the count, and
  in each pull slab the gradient rows of the other ranks.

Worst observed ratios of error to bound on an NVIDIA B200 are in DESIGN.md section 2.  ``test_comparator_*`` (no GPU)
shows that the bounds accept an fp32 emulation of the kernels' formulas and reject simulated faults.
"""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from helpers import cosine

U = 2.0 ** -24
SECOND = 1.0 + 64 * U         # second-order allowance on every first-order bound
K_GATHER, K_INV, K_DX, K_CHAIN = 9.5, 8.5, 16, 43.5
EPS = 1e-12
CLAMP32 = np.float32(1e12)    # dx_row: inv >= 1e12f <=> ||x|| <= eps
GUARD = 4096
DTYPES = {"f32": (torch.float32, 0, torch.int32), "bf16": (torch.bfloat16, 1, torch.int16),
          "f16": (torch.float16, 2, torch.int16)}
_FAKE = 0x100000              # a 1 MiB-aligned address that is never dereferenced: validation fails first


# ---------------------------------------------------------------------------------------------------------------------
# comparator (shared by the GPU tests and the CPU self-check)
# ---------------------------------------------------------------------------------------------------------------------
def _ratio(err, bound):
    err, bound = np.asarray(err, np.float64), np.asarray(bound, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err == 0, 0.0, np.inf))
    return np.where(np.isnan(r), np.inf, r)


def gather_ref(x64):
    n64 = np.linalg.norm(x64, axis=1)
    inv64 = 1.0 / np.maximum(n64, EPS)
    return x64 * inv64[:, None], inv64


def check_gather(x64, f32, inv):
    """fp32 unit rows f32 (N, C) and inverse norms inv (N,) against fp64.  Returns (failures, worst ratio)."""
    u64, inv64 = gather_ref(x64)
    f, iv = np.asarray(f32, np.float64), np.asarray(inv, np.float64)
    rf = _ratio(np.abs(f - u64), K_GATHER * U * SECOND * np.abs(u64))
    ri = _ratio(np.abs(iv - inv64), K_INV * U * SECOND * inv64)
    fails = []
    if rf.size and rf.max() > 1.0:
        r, c = np.unravel_index(int(np.argmax(rf)), rf.shape)
        fails.append(f"unit row {r} channel {c}: {f[r, c]:.9g} vs fp64 {u64[r, c]:.9g} (ratio {rf[r, c]:.3g})")
    if ri.size and ri.max() > 1.0:
        r = int(np.argmax(ri))
        fails.append(f"inv_norm row {r}: {iv[r]:.9g} vs fp64 {inv64[r]:.9g} (ratio {ri[r]:.3g})")
    worst = max(float(rf.max()) if rf.size else 0.0, float(ri.max()) if ri.size else 0.0)
    fails += _cosine_line("unit rows", f, u64, K_GATHER * U * SECOND * np.abs(u64))
    return fails, worst


def _cosine_line(what, got, ref, bound):
    """second line of evidence: a global cosine.  With |err| <= bound elementwise,
    1 - cos <= (||bound|| / ||ref||)^2."""
    nr = float(np.linalg.norm(ref))
    if nr == 0.0:
        return []
    c = cosine(got, ref)
    if not c >= 1.0 - (float(np.linalg.norm(bound)) / nr) ** 2:
        return [f"{what}: cosine {c:.15f}"]
    return []


def dx_ref(f32, inv32, g32):
    """fp64 normalisation backward on the kernel's own fp32 inputs, and the per-element scale of the bound."""
    f, g = np.asarray(f32, np.float64), np.asarray(g32, np.float64)
    inv = np.asarray(inv32, np.float64)
    dot = (f * g).sum(1)
    S = np.abs(f * g).sum(1)
    clamped = np.asarray(inv32, np.float32) >= CLAMP32
    dx = np.where(clamped[:, None], g * inv[:, None], (g - f * dot[:, None]) * inv[:, None])
    scale = inv[:, None] * (np.abs(g) + np.abs(f) * S[:, None])
    return dx, scale


def check_dx(f32, inv32, g32, dx):
    """(a) the kernel alone."""
    d64, scale = dx_ref(f32, inv32, g32)
    d = np.asarray(dx, np.float64)
    r = _ratio(np.abs(d - d64), K_DX * U * SECOND * scale)
    fails = []
    if r.size and r.max() > 1.0:
        i, c = np.unravel_index(int(np.argmax(r)), r.shape)
        fails.append(f"dx row {i} channel {c}: {d[i, c]:.9g} vs fp64 {d64[i, c]:.9g} (ratio {r[i, c]:.3g})")
    fails += _cosine_line("dx", d, d64, K_DX * U * SECOND * scale)
    return fails, float(r.max()) if r.size else 0.0


def chain_ref(x64, g32):
    """autograd derivative of F.normalize(p=2, dim=1, eps=1e-12) at x (fp64) for the gradient rows g."""
    x = torch.from_numpy(np.ascontiguousarray(x64, np.float64)).requires_grad_(True)
    torch.nn.functional.normalize(x, p=2, dim=1, eps=EPS).backward(torch.from_numpy(np.asarray(g32, np.float64)))
    u64, inv64 = gather_ref(x64)
    g = np.asarray(g32, np.float64)
    S = np.abs(u64 * g).sum(1)
    return x.grad.numpy(), inv64[:, None] * (np.abs(g) + np.abs(u64) * S[:, None])


def check_chain(x64, g32, dx):
    """(b) gather then scatter against autograd at x."""
    d64, scale = chain_ref(x64, g32)
    d = np.asarray(dx, np.float64)
    r = _ratio(np.abs(d - d64), K_CHAIN * U * SECOND * scale)
    fails = []
    if r.size and r.max() > 1.0:
        i, c = np.unravel_index(int(np.argmax(r)), r.shape)
        fails.append(f"chain dx row {i} channel {c}: {d[i, c]:.9g} vs autograd {d64[i, c]:.9g} (ratio {r[i, c]:.3g})")
    return fails, float(r.max()) if r.size else 0.0


def bf16_rne(f32):
    return torch.from_numpy(np.ascontiguousarray(f32, np.float32)).to(torch.bfloat16).view(torch.int16).numpy()


def check_bf16(f32, bf16_bits, C, N):
    """bf16 operand matrix (N_pad, C_pad) as int16 bits: RNE of the fp32 rows, zero padding columns and rows."""
    b = np.asarray(bf16_bits, np.int16)
    fails = []
    bad = int(np.count_nonzero(b[:N, :C] != bf16_rne(f32)))
    if bad:
        fails.append(f"bf16 rows: {bad} elements are not the RNE rounding of the fp32 unit row")
    if np.any(b[:N, C:] != 0):
        fails.append(f"bf16 rows: {int(np.count_nonzero(b[:N, C:]))} padding channels [C, C_pad) are not +0")
    if np.any(b[N:] != 0):
        fails.append(f"bf16 rows: {int(np.count_nonzero(b[N:]))} elements of the padding rows [N, N_pad) are not +0")
    return fails


# ---- fp32 emulation of the kernels' formulas (unfused: every product and every sum rounds) ---------------------------
def _lanes(a):
    """(N, C) -> (N, 32 lanes, 8): lane l holds channels l + 32 q, zeros beyond C."""
    N, Cc = a.shape
    z = np.zeros((N, 256), np.float32)
    z[:, :Cc] = a
    return z.reshape(N, 8, 32).transpose(0, 2, 1)


def _warp_sum(v):
    for o in (16, 8, 4, 2, 1):
        v = (v + v[:, np.arange(32) ^ o]).astype(np.float32)
    return v[:, 0]


def emulate_gather(x32):
    v = _lanes(np.asarray(x32, np.float32))
    ss = np.zeros(v.shape[:2], np.float32)
    for q in range(8):
        ss = (ss + (v[:, :, q] * v[:, :, q]).astype(np.float32)).astype(np.float32)
    ss = _warp_sum(ss)
    inv = (np.float32(1) / np.maximum(np.sqrt(ss), np.float32(1e-12))).astype(np.float32)
    return (np.asarray(x32, np.float32) * inv[:, None]).astype(np.float32), inv


def emulate_dx(f32, inv32, g32):
    f, g = np.asarray(f32, np.float32), np.asarray(g32, np.float32)
    fl, gl = _lanes(f), _lanes(g)
    dot = np.zeros(fl.shape[:2], np.float32)
    for q in range(8):
        dot = (dot + (gl[:, :, q] * fl[:, :, q]).astype(np.float32)).astype(np.float32)
    dot = _warp_sum(dot)
    inv = np.asarray(inv32, np.float32)
    proj = (g - (f * dot[:, None]).astype(np.float32)).astype(np.float32)
    return np.where((inv >= CLAMP32)[:, None], g * inv[:, None], proj * inv[:, None]).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
X_KINDS = ["normal", "small", "large", "dominant", "zero", "below_eps", "near_eps", "f16_subnormal"]
G_KINDS = ["normal", "parallel", "zero"]


def row_values(kind, C, dt, last, rs):
    base = rs.standard_normal(C)
    if kind == "normal":
        return base
    if kind == "small":
        return base * 1e-3
    if kind == "large":
        return base * 1e3
    if kind == "dominant":          # one channel carries the row (the last channel now and then)
        v = base * 1e-3
        v[C - 1 if last else rs.randint(C)] = 3.0 * rs.choice([-1.0, 1.0])
        return v
    if kind == "zero":
        return np.zeros(C)
    unit = base / max(np.linalg.norm(base), 1e-300)
    if kind == "below_eps":         # 0 < ||x|| <= eps / 4 (fp16 flushes it to a zero row)
        return unit * EPS * rs.choice([0.25, 0.1])
    if kind == "near_eps":          # ||x|| = 4 eps: small but above the clamp
        return unit * EPS * 4.0
    if kind == "f16_subnormal":     # fp16 subnormals (2^-24 .. 2^-14); the same magnitudes in the other types
        return rs.choice([-1.0, 1.0], C) * rs.randint(1, 1024, C) * 2.0 ** -24
    raise ValueError(kind)


def pixel_set(kind, n, plane, rs):
    npix = n * plane
    if kind == "ends":              # first and last pixel of every image
        return np.unique(np.concatenate([np.arange(n) * plane, np.arange(n) * plane + plane - 1]))
    if kind == "octets":            # whole octets (global 8-pixel groups), every third one
        octs = np.arange(0, npix // 8, 3)
        return (octs[:, None] * 8 + np.arange(8)).ravel()
    if kind in ("lone0", "lone7"):  # one sampled pixel in its octet, at position 0 or 7
        octs = np.arange(0, npix // 8, 2)
        return octs * 8 + (0 if kind == "lone0" else 7)
    if kind == "p18":               # cfg-2 density
        return np.sort(rs.choice(npix, max(1, int(round(0.18 * npix))), replace=False))
    if kind == "all":
        return np.arange(npix)
    if kind.startswith("n="):       # exactly N random pixels
        return np.sort(rs.choice(npix, int(kind[2:]), replace=False))
    raise ValueError(kind)


def make_inputs(C, n, plane, dt, pixset, seed, ldF=None):
    """A feature map (n, C, plane) in dtype dt with NaN at every non-sampled pixel, the sampled pixels in a random row
    order, the slot map, and fp32 gradient rows (N, ldF) with NaN in the columns [C, ldF)."""
    rs = np.random.RandomState(seed)
    pixels = pixel_set(pixset, n, plane, rs)
    N = len(pixels)
    pix = rs.permutation(pixels).astype(np.int32)               # pix[row] = global pixel id
    X = np.full((n, C, plane), np.nan)
    off = rs.randint(8)
    for r, gp in enumerate(pix):
        kind = X_KINDS[(r + off) % len(X_KINDS)]
        X[gp // plane, :, gp % plane] = row_values(kind, C, dt, r % 16 == 3, rs)
    Xt = torch.from_numpy(X).to(DTYPES[dt][0])
    x64 = Xt.double().numpy()[pix // plane, :, pix % plane] if N else np.zeros((0, C))
    slot = np.full(n * plane, -1, np.int32)
    slot[pix] = np.arange(N, dtype=np.int32)
    ldF = C if ldF is None else ldF
    g = np.full((N, ldF), np.nan, np.float32)
    u64, _ = gather_ref(x64)
    for r in range(N):
        kind = G_KINDS[(r // 2 + off) % len(G_KINDS)]
        if kind == "normal":
            g[r, :C] = rs.standard_normal(C) * rs.choice([1e-2, 1.0, 30.0])
        elif kind == "parallel":     # g || f: dx cancels to almost 0
            g[r, :C] = (u64[r] * rs.choice([-2.5, 0.7])).astype(np.float32)
        else:
            g[r, :C] = 0.0
    return types.SimpleNamespace(C=C, n=n, plane=plane, dt=dt, N=N, pix=pix, slot=slot, X=Xt, x64=x64, g=g, ldF=ldF,
                                 C_pad=(C + 63) // 64 * 64, N_pad=(N + 255) // 256 * 256, pixset=pixset)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the comparator accepts the emulation and rejects simulated faults
# ---------------------------------------------------------------------------------------------------------------------
SELF_CHECK = [(200, 2, 24, "bf16", "p18", 17), (33, 1, 375, "f32", "all", 5), (256, 5, 8, "f16", "ends", 3),
              (7, 2, 24, "bf16", "octets", 11), (129, 2, 64, "f32", "lone7", 29)]


@pytest.fixture(scope="module")
def self_check_inputs():
    return [make_inputs(*a) for a in SELF_CHECK]


def _emulated(inp):
    x32 = inp.x64.astype(np.float32)
    f, inv = emulate_gather(x32)
    return f, inv, emulate_dx(f, inv, inp.g[:, :inp.C])


def test_comparator_accepts_the_fp32_emulation(self_check_inputs):
    worst = dict(gather=0.0, dx=0.0, chain=0.0)
    for inp in self_check_inputs:
        f, inv, dx = _emulated(inp)
        fails, w = check_gather(inp.x64, f, inv)
        worst["gather"] = max(worst["gather"], w)
        assert not fails, (inp.C, inp.dt, fails)
        assert not check_bf16(f, np.pad(bf16_rne(f), ((0, inp.N_pad - inp.N), (0, inp.C_pad - inp.C))), inp.C, inp.N)
        fails, w = check_dx(f, inv, inp.g[:, :inp.C], dx)
        worst["dx"] = max(worst["dx"], w)
        assert not fails, (inp.C, inp.dt, fails)
        fails, w = check_chain(inp.x64, inp.g[:, :inp.C], dx)
        worst["chain"] = max(worst["chain"], w)
        assert not fails, (inp.C, inp.dt, fails)
    print("fp32 emulation, worst ratio to bound: " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


def _fault_gather(kind, inp):
    """what a gather with the fault returns: (x it read, its fp32 rows, its inverse norms)."""
    x32 = inp.x64.astype(np.float32)
    Xw = inp.X.float().numpy()
    b, p = inp.pix // inp.plane, inp.pix % inp.plane
    if kind == "dropped_last_channel":
        x32 = x32.copy()
        x32[:, -1] = 0.0
    elif kind == "neighbouring_pixel_in_octet":
        p2 = np.where(p % 8 == 7, p - 1, p + 1) if inp.plane > 1 else p
        x32 = Xw[b, :, np.minimum(p2, inp.plane - 1)]
    elif kind == "neighbouring_image":
        x32 = Xw[(b + 1) % inp.n, :, p]
    f, inv = emulate_gather(x32)
    if kind == "missing_eps_clamp":
        ss = np.square(x32.astype(np.float64)).sum(1)
        with np.errstate(divide="ignore", invalid="ignore"):
            inv = (1.0 / np.sqrt(ss)).astype(np.float32)
            f = (x32 * inv[:, None]).astype(np.float32)
    elif kind == "element_off_2^-18":
        f = f.copy()
        r, c = np.unravel_index(int(np.argmax(np.abs(f))), f.shape)
        f[r, c] *= np.float32(1 + 2.0 ** -18)
    return f, inv


def _fault_dx(kind, inp, f, inv):
    g = inp.g[:, :inp.C]
    if kind == "inv_norm_of_neighbouring_row":
        return emulate_dx(f, np.roll(inv, -1), g)
    if kind == "projection_on_clamped_row":
        d = emulate_dx(f, inv, g)
        proj = (g - f * (f * g).sum(1, keepdims=True)) * inv[:, None]
        return np.where((inv >= CLAMP32)[:, None], proj, d).astype(np.float32)
    if kind == "sign_error_in_f_dot":
        dot = (f.astype(np.float64) * g).sum(1, keepdims=True)
        return ((g + f * dot) * inv[:, None]).astype(np.float32)
    if kind == "element_off_2^-18":
        d = emulate_dx(f, inv, g)
        _, scale = dx_ref(f, inv, g)
        r, c = np.unravel_index(int(np.argmax(np.abs(d) / np.where(scale > 0, scale, np.inf))), d.shape)
        d[r, c] *= np.float32(1 + 2.0 ** -18)
        return d
    raise ValueError(kind)


GATHER_FAULTS = ["dropped_last_channel", "neighbouring_pixel_in_octet", "neighbouring_image", "missing_eps_clamp",
                 "element_off_2^-18"]
SCATTER_FAULTS = ["inv_norm_of_neighbouring_row", "projection_on_clamped_row", "sign_error_in_f_dot",
                  "element_off_2^-18"]
BF16_FAULTS = ["bf16_truncation", "padding_not_zeroed"]


@pytest.mark.parametrize("fault", [f"gather:{f}" for f in GATHER_FAULTS] + [f"scatter:{f}" for f in SCATTER_FAULTS] +
                         [f"bf16:{f}" for f in BF16_FAULTS])
def test_comparator_rejects_simulated_faults(fault, self_check_inputs):
    """Each fault must exceed its bound by a clear margin (ratio >= 3) on at least one input; exact checks must count
    mismatches."""
    part, kind = fault.split(":")
    ratios, msgs = [], []
    for inp in self_check_inputs:
        f0, inv0, _ = _emulated(inp)
        if part == "gather":
            if kind == "neighbouring_image" and inp.n == 1:
                continue
            f, inv = _fault_gather(kind, inp)
            with np.errstate(invalid="ignore", over="ignore"):
                fails, w = check_gather(inp.x64, f, inv)
        elif part == "scatter":
            d = _fault_dx(kind, inp, f0, inv0)
            fails, w = check_dx(f0, inv0, inp.g[:, :inp.C], d)
            fails2, w2 = check_chain(inp.x64, inp.g[:, :inp.C], d)
            fails, w = fails + fails2, max(w, w2)
        else:
            bits = np.pad(bf16_rne(f0), ((0, inp.N_pad - inp.N), (0, inp.C_pad - inp.C)))
            if kind == "bf16_truncation":
                t = (f0.view(np.int32) >> 16).astype(np.int16)
                bits[:inp.N, :inp.C] = t
            else:
                if inp.C_pad == inp.C and inp.N_pad == inp.N:
                    continue
                bits[inp.N:, :] = bf16_rne(np.ones((1, 1)))[0, 0]
                bits[:inp.N, inp.C:] = bf16_rne(np.ones((1, 1)))[0, 0]
            fails = check_bf16(f0, bits, inp.C, inp.N)
            w = float(len(fails)) * np.inf if fails else 0.0
        ratios.append(w)
        msgs.append(fails[:1])
    first = next((m for m in msgs if m), [])
    print(f"{fault}: ratio to bound per input {['%.3g' % r for r in ratios]}; first: {first}")
    assert ratios and max(ratios) >= 3.0, f"{fault}: not rejected by a clear margin ({ratios})"


# ---- validation of mscs_scatter_dense_batch (no device: the addresses are never dereferenced) -----------------------
def _lib():
    import mscs_b200
    from mscs_b200 import _lib as L
    return mscs_b200.load(), L


def _dense_item(L, **kw):
    sc = (L.ScatterItem * 1)()
    sc[0].dF = sc[0].slot = sc[0].dfeat = _FAKE
    sc[0].ldF, sc[0].n, sc[0].C, sc[0].plane = 64, 0, 64, 8
    for k, v in kw.items():
        setattr(sc[0], k, v)
    return sc


def test_dense_batch_rejects_a_misaligned_slot_map():
    """k_dense_stream reads slot entries as int4: a slot map off 16 bytes is refused.  The item has n = 0 and no rows,
    so even a library without the check would launch no block that dereferences anything."""
    lib, L = _lib()
    rows = (C.c_int32 * 1)(0)
    for off in (4, 8, 12):
        rc = lib.mscs_scatter_dense_batch(_dense_item(L, slot=_FAKE + off), rows, 1, None)
        assert rc < 0 and b"slot" in lib.mscs_last_error(), (off, rc, lib.mscs_last_error())
    for dt in (1, 2):
        rc = lib.mscs_scatter_dense_batch(_dense_item(L, slot=_FAKE + 4, dtype=dt), rows, 1, None)
        assert rc < 0 and b"slot" in lib.mscs_last_error(), (dt, rc, lib.mscs_last_error())


def test_dense_batch_rejects_2_to_the_32_elements():
    lib, L = _lib()
    rows = (C.c_int32 * 1)(0)
    for n, Cc, plane in ((1, 256, 1 << 24), (64, 256, 1 << 18), (1 << 12, 1, 1 << 20)):
        assert n * Cc * plane == 1 << 32
        rc = lib.mscs_scatter_dense_batch(_dense_item(L, n=n, C=Cc, ldF=Cc, plane=plane), rows, 1, None)
        assert rc < 0 and b"2^32" in lib.mscs_last_error(), (n, Cc, plane, rc, lib.mscs_last_error())


# ---------------------------------------------------------------------------------------------------------------------
# GPU harness: guarded buffers and the entry points
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import mscs_b200
    assert mscs_b200.load().mscs_device_ok() == 1, "libmscs.so needs a compute-capability 10.x device"
    return torch.device("cuda:0")


class Guarded:
    """A device tensor inside 4 KiB guards; tensor and guards pre-filled with 0xFF bytes (NaN in every float type)."""

    def __init__(self, shape, dtype, dev, fill=None):
        self.dtype = dtype
        self.nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        self.buf = torch.full((GUARD + self.nbytes + GUARD,), 0xFF, dtype=torch.uint8, device=dev)
        self.t = self.buf[GUARD:GUARD + self.nbytes].view(dtype).view(*shape)
        if fill is not None:
            self.t.copy_(fill)

    def ptr(self):
        return self.t.data_ptr()

    def guards_ok(self):
        return bool((self.buf[:GUARD] == 0xFF).all()) and bool((self.buf[GUARD + self.nbytes:] == 0xFF).all())

    def bits(self):
        it = {4: torch.int32, 2: torch.int16, 1: torch.uint8}[self.t.element_size()]
        return self.t.view(it)


def _ibits(t):
    return t.view({4: torch.int32, 2: torch.int16}[t.element_size()])


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _call(rc, what):
    from mscs_b200 import _lib
    if rc != 0:
        raise AssertionError(f"{what} failed ({rc}): {_lib.load().mscs_last_error().decode()}")


def _twice(run):
    """run() -> dict of Guarded outputs.  The same call twice must give the same bytes (guards included)."""
    a, b = run(), run()
    for k in a:
        assert torch.equal(a[k].buf, b[k].buf), f"{k}: two identical calls wrote different bytes"
        assert a[k].guards_ok(), f"{k}: write outside the output"
    return a


class Dev:
    """The inputs of one case on the device."""

    def __init__(self, inp, dev, n_pix=None):
        dt = DTYPES[inp.dt][0]
        self.inp = inp
        self.map = Guarded(tuple(inp.X.shape), dt, dev, inp.X)                       # NCHW, map's type
        self.map32 = Guarded(tuple(inp.X.shape), torch.float32, dev, inp.X.float())  # its exact widening
        self.nhwc = Guarded((inp.n, inp.plane, inp.C), dt, dev, inp.X.permute(0, 2, 1))
        self.nhwc32 = Guarded((inp.n, inp.plane, inp.C), torch.float32, dev, inp.X.float().permute(0, 2, 1))
        self.slot = Guarded((inp.n * inp.plane,), torch.int32, dev, torch.from_numpy(inp.slot))
        # pix holds n_pix >= N entries: rows [N, n_pix) are stale rows above a device-resident count, and hold
        # pixels that are not sampled (a kernel that reads past the count writes into them)
        n_pix = max(inp.N if n_pix is None else n_pix, 1)
        self.pix = Guarded((n_pix,), torch.int32, dev)
        self.pix.t[:inp.N] = torch.from_numpy(inp.pix)
        if n_pix > inp.N:
            free = np.flatnonzero(~sampled_mask(inp).ravel())
            assert len(free) >= n_pix - inp.N, "too few pixels for the stale rows"
            stale = np.random.RandomState(inp.N).choice(free, n_pix - inp.N, replace=False)
            self.pix.t[inp.N:] = torch.from_numpy(stale.astype(np.int32))
        self.cnt = torch.tensor([inp.N], dtype=torch.int32, device=dev)
        self.dev = dev


def gather_outputs(inp, dev, N_up=None):
    N_up = max(inp.N if N_up is None else N_up, 1)         # an empty item still needs non-null pointers
    Np = (N_up + 255) // 256 * 256
    return dict(bf16=Guarded((Np, inp.C_pad), torch.bfloat16, dev), f32=Guarded((N_up, inp.C), torch.float32, dev),
                inv=Guarded((N_up,), torch.float32, dev))


def run_gather_normalize(d):
    inp = d.inp
    o = gather_outputs(inp, d.dev)
    from mscs_b200 import _lib as L
    _call(L.load().mscs_gather_normalize(d.map32.ptr(), inp.n, inp.C, inp.plane, d.pix.ptr(), inp.N, o["bf16"].ptr(),
                                         o["f32"].ptr(), o["inv"].ptr(), _stream()), "mscs_gather_normalize")
    return o


def gather_item(it, feat, slot, cnt_ptr, o, n, Cc, plane, dtc):
    it.feat, it.n, it.C, it.plane, it.slot, it.n_rows_dev = feat, n, Cc, plane, slot, cnt_ptr
    it.anc_bf16 = o["bf16"].ptr() if "bf16" in o else None
    it.anc_f32, it.inv_norm = o["f32"].ptr(), (o["inv"].ptr() if "inv" in o else None)
    it.dtype = dtc


def run_gather_sectors(d, half):
    from mscs_b200 import _lib as L
    inp = d.inp
    o = gather_outputs(inp, d.dev)
    items = (L.GatherItem * 1)()
    gather_item(items[0], (d.map if half else d.map32).ptr(), d.slot.ptr(), d.cnt.data_ptr(), o, inp.n, inp.C,
                inp.plane, DTYPES[inp.dt][1] if half else 0)
    _call(L.load().mscs_gather_normalize_sectors_batch(items, 1, _stream()), "mscs_gather_normalize_sectors_batch")
    return o


def rows_item(it, feat, pix, cnt_ptr, rows, Cc, o, dtc, dF=None, ldF=0, dfeat=None):
    it.feat, it.pix, it.n_rows_dev, it.rows, it.C = feat, pix, cnt_ptr, rows, Cc
    it.anc_bf16 = o["bf16"].ptr() if o and "bf16" in o else None
    it.anc_f32 = o["f32"].ptr() if o and "f32" in o else None
    it.inv_norm = o["inv"].ptr() if o and "inv" in o else None
    it.dF, it.ldF, it.dfeat, it.dtype = dF, ldF, dfeat, dtc


def run_gather_rows(d, half, dev_count=False):
    from mscs_b200 import _lib as L
    inp = d.inp
    o = gather_outputs(inp, d.dev)
    items = (L.RowsItem * 1)()
    rows_item(items[0], (d.nhwc if half else d.nhwc32).ptr(), d.pix.ptr(), d.cnt.data_ptr() if dev_count else None,
              inp.N, inp.C, o, DTYPES[inp.dt][1] if half else 0)
    _call(L.load().mscs_gather_rows_nhwc_batch(items, 1, _stream()), "mscs_gather_rows_nhwc_batch")
    return o


def p2p_slabs(world, nbytes_each, off, dev):
    return [Guarded((off + nbytes_each,), torch.uint8, dev) for _ in range(world)]


def slab_view(slab, off, shape, dtype):
    nb = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    return slab.t[off:off + nb].view(dtype).view(*shape)


P2P_OFF = 512            # byte offset of the operand matrix / gradient rows inside a slab


def run_gather_rows_p2p(d, half, world=1, rank=0, slabs=None, pix=None, feat=None, o=None, dev_count=False):
    from mscs_b200 import _lib as L
    inp = d.inp
    o = gather_outputs(inp, d.dev) if o is None else o
    nb = inp.N_pad * inp.C_pad * 2
    slabs = p2p_slabs(world, nb, P2P_OFF, d.dev) if slabs is None else slabs
    ptrs = L.ptr_array([s.ptr() for s in slabs])
    feat = (d.nhwc if half else d.nhwc32).ptr() if feat is None else feat
    _call(L.load().mscs_gather_rows_p2p(feat, inp.C, d.pix.ptr() if pix is None else pix, inp.N,
                                        d.cnt.data_ptr() if dev_count else None, ptrs, world, rank, P2P_OFF,
                                        o["f32"].ptr(), o["inv"].ptr(), _stream(),
                                        DTYPES[inp.dt][1] if half else 0), "mscs_gather_rows_p2p")
    return dict(f32=o["f32"], inv=o["inv"], **{f"slab{r}": s for r, s in enumerate(slabs)})


def run_gather_p2p(d, half, world=1, rank=0, slabs=None, slot=None, feat=None, n=None, o=None):
    from mscs_b200 import _lib as L
    inp = d.inp
    o = gather_outputs(inp, d.dev) if o is None else o
    nb = inp.N_pad * inp.C_pad * 2
    slabs = p2p_slabs(world, nb, P2P_OFF, d.dev) if slabs is None else slabs
    ptrs = L.ptr_array([s.ptr() for s in slabs])
    _call(L.load().mscs_gather_normalize_p2p((d.map if half else d.map32).ptr() if feat is None else feat,
                                             inp.n if n is None else n, inp.C, inp.plane,
                                             d.slot.ptr() if slot is None else slot, inp.N, None, ptrs, world, rank,
                                             P2P_OFF, o["f32"].ptr(), o["inv"].ptr(), _stream(),
                                             DTYPES[inp.dt][1] if half else 0), "mscs_gather_normalize_p2p")
    return dict(f32=o["f32"], inv=o["inv"], **{f"slab{r}": s for r, s in enumerate(slabs)})


def run_gather_raw(d, half, nhwc):
    from mscs_b200 import _lib as L
    inp = d.inp
    o = dict(f32=Guarded((max(inp.N, 1), inp.C), torch.float32, d.dev))
    dtc = DTYPES[inp.dt][1] if half else 0
    if nhwc:
        items = (L.RowsItem * 1)()
        rows_item(items[0], (d.nhwc if half else d.nhwc32).ptr(), d.pix.ptr(), None, inp.N, inp.C, o, dtc)
        _call(L.load().mscs_gather_raw_rows_batch(items, 1, _stream()), "mscs_gather_raw_rows_batch")
    else:
        items = (L.GatherItem * 1)()
        gather_item(items[0], (d.map if half else d.map32).ptr(), d.slot.ptr(), None, o, inp.n, inp.C, inp.plane,
                    dtc)
        _call(L.load().mscs_gather_raw_batch(items, 1, _stream()), "mscs_gather_raw_batch")
    return o


# ---- scatters: inputs are the fp32 unit rows / inverse norms of a gather, and dF (N, ldF) ---------------------------
def dF_dev(inp, dev, N_up=None):
    N_up = max(inp.N if N_up is None else N_up, 1)
    g = torch.full((N_up, inp.ldF), float("nan"))
    g[:inp.N] = torch.from_numpy(inp.g)
    return Guarded((N_up, inp.ldF), torch.float32, dev, g)


def run_scatter_grad(d, f32, inv, zero_fill):
    from mscs_b200 import _lib as L
    inp = d.inp
    dF = dF_dev(inp, d.dev)
    out = Guarded((inp.n, inp.C, inp.plane), torch.float32, d.dev)
    _call(L.load().mscs_scatter_grad(dF.ptr(), inp.ldF, f32.ptr(), inv.ptr(), d.pix.ptr(), inp.N, inp.n, inp.C,
                                     inp.plane, out.ptr(), zero_fill, _stream()), "mscs_scatter_grad")
    return dict(out=out, dF=dF)


def scatter_item(it, dF, ldF, f32, inv, slot, n, Cc, plane, dfeat, dtc, cnt_ptr=None):
    it.dF, it.ldF, it.anc_f32, it.inv_norm, it.slot = dF, ldF, f32, inv, slot
    it.n, it.C, it.plane, it.dfeat, it.dtype, it.n_rows_dev = n, Cc, plane, dfeat, dtc, cnt_ptr


def run_scatter_sectors(d, f32, inv):
    from mscs_b200 import _lib as L
    inp = d.inp
    dF = dF_dev(inp, d.dev)
    out = Guarded((inp.n, inp.C, inp.plane), torch.float32, d.dev)
    items = (L.ScatterItem * 1)()
    scatter_item(items[0], dF.ptr(), inp.ldF, f32.ptr(), inv.ptr(), d.slot.ptr(), inp.n, inp.C, inp.plane, out.ptr(), 0)
    _call(L.load().mscs_scatter_sectors_batch(items, 1, _stream()), "mscs_scatter_sectors_batch")
    return dict(out=out, dF=dF)


def run_scatter_dense(d, f32, inv, half, raw=False, dev_count=False, N_up=None):
    from mscs_b200 import _lib as L
    inp = d.inp
    dF = dF_dev(inp, d.dev, N_up)
    out = Guarded((inp.n, inp.C, inp.plane), DTYPES[inp.dt][0] if half else torch.float32, d.dev)
    items = (L.ScatterItem * 1)()
    scatter_item(items[0], dF.ptr(), inp.ldF, None if raw else f32.ptr(), None if raw else inv.ptr(), d.slot.ptr(),
                 inp.n, inp.C, inp.plane, out.ptr(), DTYPES[inp.dt][1] if half else 0,
                 d.cnt.data_ptr() if dev_count else None)
    rows = (C.c_int32 * 1)(inp.N if N_up is None else N_up)
    _call(L.load().mscs_scatter_dense_batch(items, rows, 1, _stream()), "mscs_scatter_dense_batch")
    return dict(out=out, dF=dF)


def run_scatter_rows(d, f32, inv, half, raw=False, dev_count=False, N_up=None):
    from mscs_b200 import _lib as L
    inp = d.inp
    dF = dF_dev(inp, d.dev, N_up)
    out = Guarded((inp.n, inp.plane, inp.C), DTYPES[inp.dt][0] if half else torch.float32, d.dev)
    items = (L.RowsItem * 1)()
    o = None if raw else dict(f32=f32, inv=inv)
    rows_item(items[0], None, d.pix.ptr(), d.cnt.data_ptr() if dev_count else None,
              inp.N if N_up is None else N_up, inp.C, o, DTYPES[inp.dt][1] if half else 0, dF.ptr(), inp.ldF, out.ptr())
    _call(L.load().mscs_scatter_rows_nhwc_batch(items, 1, _stream()), "mscs_scatter_rows_nhwc_batch")
    return dict(out=out, dF=dF)


def pull_slabs(inp, world, rpr, dev):
    """one slab per rank with the gradient rows at P2P_OFF; only rank r's rows [r rpr, (r+1) rpr) are valid, the
    others are NaN (a read from the wrong rank turns the dx row into NaN)."""
    slabs = []
    for r in range(world):
        s = Guarded((P2P_OFF + max(inp.N, 1) * inp.ldF * 4,), torch.uint8, dev)
        v = slab_view(s, P2P_OFF, (max(inp.N, 1), inp.ldF), torch.float32)
        lo, hi = r * rpr, min(inp.N, (r + 1) * rpr)
        if hi > lo:
            v[lo:hi] = torch.from_numpy(inp.g[lo:hi]).to(dev)
        slabs.append(s)
    return slabs


def run_pull(d, f32, inv, half, nhwc, world=1, rpr=None, slabs=None, slot=None, pix=None, n=None, N=None):
    from mscs_b200 import _lib as L
    inp = d.inp
    rpr = max(128, (inp.N + 127) // 128 * 128) if rpr is None else rpr
    slabs = pull_slabs(inp, world, rpr, d.dev) if slabs is None else slabs
    ptrs = L.ptr_array([s.ptr() for s in slabs])
    n = inp.n if n is None else n
    dt = DTYPES[inp.dt][0] if half else torch.float32
    dtc = DTYPES[inp.dt][1] if half else 0
    if nhwc:
        out = Guarded((n, inp.plane, inp.C), dt, d.dev)
        _call(L.load().mscs_scatter_rows_pull(ptrs, world, P2P_OFF, rpr, inp.ldF, f32.ptr(), inv.ptr(),
                                              d.pix.ptr() if pix is None else pix, inp.N if N is None else N, inp.C,
                                              out.ptr(), _stream(), dtc), "mscs_scatter_rows_pull")
    else:
        out = Guarded((n, inp.C, inp.plane), dt, d.dev)
        _call(L.load().mscs_scatter_sectors_pull(ptrs, world, P2P_OFF, rpr, inp.ldF, f32.ptr(), inv.ptr(),
                                                 d.slot.ptr() if slot is None else slot, n, inp.C, inp.plane,
                                                 out.ptr(), _stream(), dtc), "mscs_scatter_sectors_pull")
    return dict(out=out, **{f"slab{r}": s for r, s in enumerate(slabs)})


# ---- what each output must hold ------------------------------------------------------------------------------------
def _host(t):
    return t.detach().cpu()


def sampled_mask(inp):
    m = np.zeros(inp.n * inp.plane, bool)
    m[inp.pix] = True
    return m.reshape(inp.n, inp.plane)


def octet_mask(inp):
    """pixels in a (global) 8-pixel octet that holds a sampled pixel"""
    m = sampled_mask(inp).ravel()
    o = m.reshape(-1, 8).any(1) if m.size % 8 == 0 else None
    return np.repeat(o, 8).reshape(inp.n, inp.plane)


def nchw_rows(out, inp):
    """(N, C) values of an NCHW output at the sampled pixels, in row order"""
    t = _host(out)
    return t[torch.from_numpy(inp.pix // inp.plane).long(), :, torch.from_numpy(inp.pix % inp.plane).long()]


def nhwc_rows(out, inp):
    t = _host(out).reshape(inp.n * inp.plane, inp.C)
    return t[torch.from_numpy(inp.pix).long()]


def assert_nchw_extent(out, inp, written):
    """written: (n, plane) bool of the pixels the entry point may write (all C channels); the rest must be the
    pre-fill; the written non-sampled pixels must be +0."""
    bits = _ibits(_host(out))
    w = torch.from_numpy(written)[:, None, :].expand(inp.n, inp.C, inp.plane)
    assert bool((bits[~w] == -1).all()), f"{int((bits[~w] != -1).sum())} elements outside the promised extent written"
    zero = torch.from_numpy(written & ~sampled_mask(inp))[:, None, :].expand(inp.n, inp.C, inp.plane)
    assert bool((bits[zero] == 0).all()), "pixels next to the sampled ones are not explicit +0"


def assert_nhwc_extent(out, inp):
    bits = _ibits(_host(out)).reshape(inp.n * inp.plane, inp.C)
    keep = torch.from_numpy(~sampled_mask(inp).ravel())
    assert bool((bits[keep] == -1).all()), "channels-last scatter wrote a non-sampled pixel"


def as_dtype_bits(dx32, dt):
    return _ibits(torch.as_tensor(dx32).to(DTYPES[dt][0]))


# ---------------------------------------------------------------------------------------------------------------------
# the case matrix of the single-item tests
# ---------------------------------------------------------------------------------------------------------------------
CHANNELS = [1, 7, 8, 31, 32, 33, 63, 64, 65, 127, 128, 129, 192, 200, 255, 256]
# (plane, n, pixel set) cycled against the channel counts; planes 4 / 12 take the fp32 dense writer and the unbatched
# paths only, 1 and 375 (15 x 25) the unbatched host path, 8192 = 64 x 128
GEOMS = [(8, 1, "all"), (24, 2, "ends"), (375, 2, "p18"), (8192, 1, "p18"), (24, 5, "lone0"), (8, 5, "octets"),
         (12, 2, "all"), (4, 5, "ends"), (1, 5, "all"), (24, 2, "lone7"), (8192, 2, "octets"), (375, 1, "ends"),
         (24, 5, "p18"), (8, 2, "lone7"), (4, 2, "all"), (8192, 1, "lone0")]
CASES = {}
for _i, _C in enumerate(CHANNELS):
    for _j, _dt in enumerate(("f32", "bf16", "f16")):
        _plane, _n, _ps = GEOMS[(_i + 5 * _j) % len(GEOMS)]
        _ld = _C + (0 if (_i + _j) % 3 == 0 else 3 + 8 * _j)
        CASES[f"c{_C}_p{_plane}_n{_n}_{_ps}_{_dt}_ld{_ld}"] = (_C, _n, _plane, _dt, _ps, 1000 + 31 * _i + _j, _ld)


def test_case_matrix_covers_every_axis():
    v = list(CASES.values())
    assert {c[0] for c in v} == set(CHANNELS)
    assert {(c[0] + 63) // 64 for c in v} == {1, 2, 3, 4}
    assert {c[2] for c in v} == {1, 4, 8, 12, 24, 375, 8192}
    assert {c[1] for c in v} == {1, 2, 5}
    assert {c[4] for c in v} == {"ends", "octets", "lone0", "lone7", "p18", "all"}
    assert any(c[6] > c[0] for c in v) and any(c[6] == c[0] for c in v)
    for dt in DTYPES:        # every type meets planes that are and are not a multiple of 8
        assert {c[2] % 8 == 0 for c in v if c[3] == dt} == {True, False}


_WORST = {}


def _worst(name, r):
    _WORST[name] = max(_WORST.get(name, 0.0), r)


def _report():
    print("worst ratio to bound: " + ", ".join(f"{k} {v:.3f}" for k, v in sorted(_WORST.items())))


def check_gather_outputs(name, o, inp, ref_f32=None):
    """fp64 bound, bf16 = RNE, padding zero, guards; returns host (f32, inv, bf16 bits)."""
    for k, g in o.items():
        assert g.guards_ok(), f"{name}: {k} written outside its buffer"
    f, iv = _host(o["f32"].t).numpy(), _host(o["inv"].t).numpy()
    fails, w = check_gather(inp.x64, f, iv)
    _worst(name, w)
    assert not fails, f"{name}: " + "; ".join(fails)
    if "bf16" in o:
        bits = _host(o["bf16"].bits()).numpy()
        fails = check_bf16(f, bits, inp.C, inp.N)
        assert not fails, f"{name}: " + "; ".join(fails)
        return f, iv, bits
    return f, iv, None


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_row_kernels_vs_fp64(name, dev):
    Cc, n, plane, dt, ps, seed, ld = CASES[name]
    inp = make_inputs(Cc, n, plane, dt, ps, seed, ld)
    d = Dev(inp, dev)
    half = dt != "f32"
    sectors = plane % 8 == 0
    # ---- gathers: the fp64 bound, then bit-identical rows across kernels and between a half map and its widening
    ref = _twice(lambda: run_gather_normalize(d))
    f, iv, bits = check_gather_outputs("mscs_gather_normalize", ref, inp)
    same = [("mscs_gather_rows_nhwc_batch fp32", _twice(lambda: run_gather_rows(d, False))),
            ("mscs_gather_rows_p2p fp32", _twice(lambda: run_gather_rows_p2p(d, False)))]
    if half:
        same += [(f"mscs_gather_rows_nhwc_batch {dt}", _twice(lambda: run_gather_rows(d, True))),
                 (f"mscs_gather_rows_p2p {dt}", _twice(lambda: run_gather_rows_p2p(d, True)))]
    if sectors:
        same += [("mscs_gather_normalize_sectors_batch fp32", _twice(lambda: run_gather_sectors(d, False)))]
        if half:
            same += [(f"mscs_gather_normalize_sectors_batch {dt}", _twice(lambda: run_gather_sectors(d, True)))]
    for tag, o in same:
        for k, g in o.items():
            assert g.guards_ok(), f"{tag}: {k} written outside its buffer"
        _worst(tag.split()[0], check_gather(inp.x64, _host(o["f32"].t).numpy(), _host(o["inv"].t).numpy())[1])
        assert torch.equal(_host(o["f32"].bits()), _host(ref["f32"].bits())), f"{tag}: fp32 rows differ"
        assert torch.equal(_host(o["inv"].bits()), _host(ref["inv"].bits())), f"{tag}: inv_norm differs"
        b = o["bf16"].bits() if "bf16" in o else slab_view(o["slab0"], P2P_OFF, (inp.N_pad, inp.C_pad), torch.int16)
        assert torch.equal(_host(b), _host(ref["bf16"].bits())), f"{tag}: bf16 rows differ"
    if sectors:
        for h in ((False, True) if half else (False,)):
            o = _twice(lambda: run_gather_p2p(d, h))
            tag = f"k_gather_p2p {dt if h else 'fp32'}"
            o["bf16"] = types.SimpleNamespace(bits=lambda: slab_view(o["slab0"], P2P_OFF, (inp.N_pad, inp.C_pad),
                                                                        torch.int16), guards_ok=o["slab0"].guards_ok)
            check_gather_outputs("mscs_gather_normalize_p2p", o, inp)
            if h:
                assert torch.equal(_host(o["f32"].bits()), _host(p2p32["f32"].bits())), f"{tag}: half != widening"
            else:
                p2p32 = o
    # raw gathers: x.float() at the sampled pixels, exactly
    want_raw = torch.from_numpy(inp.x64.astype(np.float32))
    for nhwc in (False, True):
        if not nhwc and not sectors:
            continue
        for h in ((False, True) if half else (False,)):
            o = _twice(lambda: run_gather_raw(d, h, nhwc))
            assert torch.equal(_ibits(_host(o["f32"].t)), _ibits(want_raw)), f"raw gather (nhwc={nhwc}, half={h})"
            _worst("mscs_gather_raw_rows_batch (exact)" if nhwc else "mscs_gather_raw_batch (exact)", 0.0)

    # ---- scatters on the production inputs: the fp32 rows and inverse norms of the gather
    f32, inv = ref["f32"], ref["inv"]
    g = inp.g[:, :Cc]
    o = _twice(lambda: run_scatter_grad(d, f32, inv, 0))
    assert_nchw_extent(o["out"].t, inp, sampled_mask(inp))
    dx = nchw_rows(o["out"].t, inp)
    fails, wdx = check_dx(f, iv, g, dx.numpy())
    _worst("mscs_scatter_grad", wdx)
    assert not fails, "k_scatter_grad: " + "; ".join(fails)
    fails, w = check_chain(inp.x64, g, dx.numpy())
    _worst("chain (gather + scatter vs autograd)", w)
    assert not fails, "; ".join(fails)
    dxb = _ibits(dx)
    o = _twice(lambda: run_scatter_grad(d, f32, inv, 1))
    assert torch.equal(_ibits(nchw_rows(o["out"].t, inp)), dxb), "mscs_scatter_grad zero_fill=1: dx differs"
    assert_nchw_extent(o["out"].t, inp, np.ones((n, plane), bool))
    if sectors:
        o = _twice(lambda: run_scatter_sectors(d, f32, inv))
        assert_nchw_extent(o["out"].t, inp, octet_mask(inp))
        assert torch.equal(_ibits(nchw_rows(o["out"].t, inp)), dxb), "k_scatter_sectors_batch: dx differs"
        _worst("mscs_scatter_sectors_batch", wdx)      # bit-identical dx: the same ratio
    dense_types = [False] + ([True] if half and sectors else [])
    if plane % 4 == 0:
        for h in dense_types:
            o = _twice(lambda: run_scatter_dense(d, f32, inv, h))
            bits = _ibits(_host(o["out"].t))
            assert bool((bits != -1).all()), "dense writer left elements unwritten"
            got = _ibits(nchw_rows(o["out"].t, inp))
            want = as_dtype_bits(dx, dt) if h else dxb
            assert torch.equal(got, want), f"k_dense_stream (half={h}): dx differs"
            assert int(torch.count_nonzero(bits)) == int(torch.count_nonzero(want)), "dense writer: non-zero elsewhere"
            # k_dx_rows: dF rows [0, N), columns [0, C) hold dx in place; columns [C, ldF) untouched
            dFb = _host(o["dF"].bits())
            assert torch.equal(dFb[:, :Cc], dxb), "k_dx_rows: dx in dF differs"
            _worst("mscs_scatter_dense_batch", wdx)
            assert bool(torch.isnan(_host(o["dF"].t[:, Cc:])).all()), "k_dx_rows wrote columns [C, ldF)"
            # raw item: dF stored as it is
            o = _twice(lambda: run_scatter_dense(d, None, None, h, raw=True))
            want = as_dtype_bits(torch.from_numpy(g.copy()), dt) if h else _ibits(torch.from_numpy(g.copy()))
            assert torch.equal(_ibits(nchw_rows(o["out"].t, inp)), want), f"raw dense item (half={h})"
            assert int(torch.count_nonzero(_ibits(_host(o["out"].t)))) == int(torch.count_nonzero(want))
    for h in ((False, True) if half else (False,)):
        want = as_dtype_bits(dx, dt) if h else dxb
        o = _twice(lambda: run_scatter_rows(d, f32, inv, h))
        assert_nhwc_extent(o["out"].t, inp)
        assert torch.equal(_ibits(nhwc_rows(o["out"].t, inp)), want), f"k_scatter_rows_nhwc (half={h}): dx differs"
        _worst("mscs_scatter_rows_nhwc_batch", wdx)
        o = _twice(lambda: run_scatter_rows(d, None, None, h, raw=True))
        assert_nhwc_extent(o["out"].t, inp)
        wr = as_dtype_bits(torch.from_numpy(g.copy()), dt) if h else _ibits(torch.from_numpy(g.copy()))
        assert torch.equal(_ibits(nhwc_rows(o["out"].t, inp)), wr), f"raw rows item (half={h})"
        o = _twice(lambda: run_pull(d, f32, inv, h, nhwc=True))
        assert_nhwc_extent(o["out"].t, inp)
        assert torch.equal(_ibits(nhwc_rows(o["out"].t, inp)), want), f"k_scatter_rows_pull (half={h}): dx differs"
        _worst("mscs_scatter_rows_pull", wdx)
        if sectors:
            o = _twice(lambda: run_pull(d, f32, inv, h, nhwc=False))
            assert_nchw_extent(o["out"].t, inp, octet_mask(inp))
            assert torch.equal(_ibits(nchw_rows(o["out"].t, inp)), want), f"k_scatter_sectors_pull (half={h})"
            _worst("mscs_scatter_sectors_pull", wdx)
    print(f"[{name}] N={inp.N} C_pad={inp.C_pad}")
    _report()


@pytest.mark.gpu
@pytest.mark.parametrize("plane", [4, 12])
def test_half_and_sector_paths_reject_planes_that_are_not_octets(plane, dev):
    """planes of 4 / 12 pixels: the fp32 dense writer takes them (test_row_kernels_vs_fp64), the half dense writer and
    every sector path refuse them before any launch.  No call here could touch memory outside its buffers even if the
    check it tests were gone: the scatters get n = 0 images and 0 rows (k_dx_rows returns on the row bound, the writers
    get no blocks), and the gathers, which need n >= 1, get every buffer at the size of the case (their loads are
    scalar, and they store only rows the slot map names, 16-byte stores at 16-byte aligned row starts)."""
    from mscs_b200 import _lib as L
    lib = L.load()
    inp = make_inputs(64, 2, plane, "bf16", "all", 7)
    d = Dev(inp, dev)
    o = gather_outputs(inp, dev)
    dF = dF_dev(inp, dev)
    slabs = pull_slabs(inp, 1, 128, dev)
    outs = [Guarded((inp.n, inp.C, plane), t, dev) for t in (torch.bfloat16, torch.float16, torch.float32)]
    before = dict(dF=dF.buf.clone(), slab=slabs[0].buf.clone())
    rejected = lambda rc, what: (rc < 0 and b"plane" in lib.mscs_last_error(), what, rc, lib.mscs_last_error())
    for dtc, out in ((1, outs[0]), (2, outs[1])):
        items = (L.ScatterItem * 1)()
        scatter_item(items[0], dF.ptr(), inp.ldF, o["f32"].ptr(), o["inv"].ptr(), d.slot.ptr(), 0, 64, plane,
                     out.ptr(), dtc)
        r = rejected(lib.mscs_scatter_dense_batch(items, (C.c_int32 * 1)(0), 1, None), "half dense writer")
        assert r[0], r
        r = rejected(lib.mscs_scatter_sectors_pull(L.ptr_array([slabs[0].ptr()]), 1, P2P_OFF, 128, inp.ldF,
                                                   o["f32"].ptr(), o["inv"].ptr(), d.slot.ptr(), 0, 64, plane,
                                                   out.ptr(), None, dtc), "half pull scatter")
        assert r[0], r
    items = (L.ScatterItem * 1)()
    scatter_item(items[0], dF.ptr(), inp.ldF, o["f32"].ptr(), o["inv"].ptr(), d.slot.ptr(), 0, 64, plane,
                 outs[2].ptr(), 0)
    r = rejected(lib.mscs_scatter_sectors_batch(items, 1, None), "sector scatter")
    assert r[0], r
    items = (L.GatherItem * 1)()
    gather_item(items[0], d.map.ptr(), d.slot.ptr(), d.cnt.data_ptr(), o, inp.n, 64, plane, 1)
    r = rejected(lib.mscs_gather_normalize_sectors_batch(items, 1, None), "sector gather")
    assert r[0], r
    r = rejected(lib.mscs_gather_raw_batch(items, 1, None), "raw sector gather")
    assert r[0], r
    r = rejected(lib.mscs_gather_normalize_p2p(d.map32.ptr(), inp.n, 64, plane, d.slot.ptr(), inp.N, None,
                                               L.ptr_array([o["bf16"].ptr()]), 1, 0, 0, o["f32"].ptr(),
                                               o["inv"].ptr(), None, 0), "p2p gather")
    assert r[0], r
    torch.cuda.synchronize()
    for k, g in list(o.items()) + [(f"out{i}", g) for i, g in enumerate(outs)]:
        assert bool((g.buf == 0xFF).all()), f"{k} written by a refused call"
    assert torch.equal(dF.buf, before["dF"]) and torch.equal(slabs[0].buf, before["slab"]), \
        "dF written by a refused call"


# ---------------------------------------------------------------------------------------------------------------------
# row counts: host counts, device counts with stale rows above, zero
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 255, 256, 257])
@pytest.mark.parametrize("mode", ["host", "device"])
def test_row_counts(N, mode, dev):
    """Row counts at and one off the 256-row padding.  Device mode: the upper bound is 300 rows above the count, and the
    rows in between are stale: the outputs hold the pre-fill there, dF, the unit rows and the inverse norms hold NaN,
    and pix holds pixels that are not sampled.  Nothing at or above the count may be written, except the bf16 padding
    rows up to the count rounded to 256; a scatter that passes the count stores into those pixels."""
    inp = make_inputs(65, 2, 24 * 16, "bf16", f"n={N}", 4242 + N, ldF=72)
    up = N + 300 if mode == "device" else N
    dc = mode == "device"
    d = Dev(inp, dev, n_pix=up)
    from mscs_b200 import _lib as L
    lib = L.load()
    # gathers with the count in device memory (sectors: always; rows and rows-p2p: in device mode) and an upper bound
    for kind in ("sectors", "rows", "rows_p2p"):
        o = gather_outputs(inp, dev, up)
        if kind == "sectors":
            items = (L.GatherItem * 1)()
            gather_item(items[0], d.map.ptr(), d.slot.ptr(), d.cnt.data_ptr(), o, inp.n, inp.C, inp.plane, 1)
            _call(lib.mscs_gather_normalize_sectors_batch(items, 1, _stream()), kind)
            bits = o["bf16"].bits()
        elif kind == "rows":
            items = (L.RowsItem * 1)()
            rows_item(items[0], d.nhwc.ptr(), d.pix.ptr(), d.cnt.data_ptr() if dc else None, up, inp.C, o, 1)
            _call(lib.mscs_gather_rows_nhwc_batch(items, 1, _stream()), kind)
            bits = o["bf16"].bits()
        else:
            slab = Guarded((P2P_OFF + ((up + 255) // 256 * 256) * inp.C_pad * 2,), torch.uint8, dev)
            _call(lib.mscs_gather_rows_p2p(d.nhwc.ptr(), inp.C, d.pix.ptr(), up, d.cnt.data_ptr() if dc else None,
                                           L.ptr_array([slab.ptr()]), 1, 0, P2P_OFF, o["f32"].ptr(), o["inv"].ptr(),
                                           _stream(), 1), kind)
            bits = slab_view(slab, P2P_OFF, ((up + 255) // 256 * 256, inp.C_pad), torch.int16)
        torch.cuda.synchronize()
        f, iv = _host(o["f32"].t[:N]).numpy(), _host(o["inv"].t[:N]).numpy()
        fails, w = check_gather(inp.x64, f, iv)
        _worst(f"counts gather {kind}", w)
        assert not fails, f"{kind}: {fails}"
        b = _host(bits)
        assert not check_bf16(f, b[:inp.N_pad], inp.C, N), kind
        assert bool((b[inp.N_pad:] == -1).all()), f"{kind}: bf16 rows at or above the padded count written"
        assert bool((_host(o["f32"].bits()[N:]) == -1).all()) and bool((_host(o["inv"].bits()[N:]) == -1).all()), \
            f"{kind}: fp32 rows / inv_norm at or above the count written"
    # scatters with an upper bound: unit rows, inverse norms and dF allocated for `up` rows, NaN above the count
    o = gather_outputs(inp, dev, up)
    _call(lib.mscs_gather_normalize(d.map32.ptr(), inp.n, inp.C, inp.plane, d.pix.ptr(), N, o["bf16"].ptr(),
                                    o["f32"].ptr(), o["inv"].ptr(), _stream()), "mscs_gather_normalize")
    want = run_scatter_grad(d, o["f32"], o["inv"], 0)
    dxb = _ibits(nchw_rows(want["out"].t, inp))
    raw = _ibits(torch.from_numpy(np.ascontiguousarray(inp.g[:, :inp.C])).to(torch.bfloat16))
    for h in (False, True):
        s = run_scatter_dense(d, o["f32"], o["inv"], h, dev_count=dc, N_up=up)
        got = _ibits(nchw_rows(s["out"].t, inp))
        assert torch.equal(got, as_dtype_bits(nchw_rows(want["out"].t, inp), "bf16") if h else dxb), "dense"
        assert torch.equal(_host(s["dF"].bits()[:N, :inp.C]), dxb), "k_dx_rows"
        assert bool(torch.isnan(_host(s["dF"].t[N:])).all()), "k_dx_rows wrote rows at or above the count"
        assert s["out"].guards_ok() and s["dF"].guards_ok()
        # channels-last, normalised and raw items: only the N sampled pixels are written (the stale pixels of rows
        # [N, up) are not sampled, so assert_nhwc_extent sees a store past the count)
        for is_raw in (False, True):
            s = run_scatter_rows(d, o["f32"], o["inv"], h, raw=is_raw, dev_count=dc, N_up=up)
            assert_nhwc_extent(s["out"].t, inp)
            wr = (raw if h else _ibits(torch.from_numpy(np.ascontiguousarray(inp.g[:, :inp.C])))) if is_raw else \
                (as_dtype_bits(nchw_rows(want["out"].t, inp), "bf16") if h else dxb)
            assert torch.equal(_ibits(nhwc_rows(s["out"].t, inp)), wr), f"rows scatter (raw={is_raw}, half={h})"
            assert s["out"].guards_ok() and s["dF"].guards_ok()
    _report()


@pytest.mark.gpu
@pytest.mark.parametrize("Cc", [33, 256])
def test_rows_owned_by_another_rank(Cc, dev):
    """pix < 0 (pooled mode: the row belongs to another rank).  k_gather_normalize and k_gather_rows_nhwc zero that
    row's bf16 operand row and leave its fp32 row and inv_norm alone; k_scatter_grad and k_scatter_rows_nhwc write
    nothing for it (its pixel keeps the pre-fill, or the zero of zero_fill); every other row is the row of the call
    in which no row is foreign, bit for bit."""
    from mscs_b200 import _lib as L
    lib = L.load()
    inp = make_inputs(Cc, 2, 375, "f32", "p18", 555 + Cc, Cc + 3)
    d = Dev(inp, dev)
    full = run_gather_normalize(d)
    full_rows = run_gather_rows(d, False)
    full_dx = _ibits(nchw_rows(run_scatter_grad(d, full["f32"], full["inv"], 0)["out"].t, inp))
    foreign = np.arange(inp.N) % 5 == 2
    own = torch.from_numpy(~foreign)
    d.pix.t[:inp.N] = torch.from_numpy(np.where(foreign, -1, inp.pix).astype(np.int32))
    lost = np.zeros((inp.n, inp.plane), bool)                 # the pixels of the foreign rows
    lost.ravel()[inp.pix[foreign]] = True
    for tag, o in (("k_gather_normalize", run_gather_normalize(d)), ("k_gather_rows_nhwc", run_gather_rows(d, False))):
        ref = full if tag == "k_gather_normalize" else full_rows
        for k in o:
            assert o[k].guards_ok(), f"{tag}: {k}"
        b = _host(o["bf16"].bits())
        assert bool((b[:inp.N][torch.from_numpy(foreign)] == 0).all()), f"{tag}: bf16 row of a pix < 0 row is not +0"
        assert torch.equal(b[:inp.N][own], _host(ref["bf16"].bits())[:inp.N][own]), f"{tag}: bf16 rows"
        assert bool((b[inp.N:] == 0).all()), f"{tag}: padding rows"
        for k in ("f32", "inv"):
            got = _host(o[k].bits())
            assert bool((got[torch.from_numpy(foreign)] == -1).all()), f"{tag}: {k} of a pix < 0 row written"
            assert torch.equal(got[own], _host(ref[k].bits())[own]), f"{tag}: {k} of the own rows"
    # the scatters get the full fp32 rows and inverse norms: a foreign row would have a valid dx, but must not store it
    for zero_fill in (0, 1):
        o = run_scatter_grad(d, full["f32"], full["inv"], zero_fill)
        assert o["out"].guards_ok()
        bits = _ibits(_host(o["out"].t))
        m = torch.from_numpy(lost)[:, None, :].expand(inp.n, Cc, inp.plane)
        assert bool((bits[m] == (0 if zero_fill else -1)).all()), f"zero_fill={zero_fill}: pixel of a pix < 0 row"
        assert torch.equal(_ibits(nchw_rows(o["out"].t, inp))[own], full_dx[own]), f"zero_fill={zero_fill}: own rows"
    o = run_scatter_rows(d, full["f32"], full["inv"], False)
    rows_bits = _ibits(_host(o["out"].t)).reshape(inp.n * inp.plane, Cc)
    assert bool((rows_bits[torch.from_numpy(inp.pix[foreign]).long()] == -1).all()), "rows scatter: foreign pixel"
    assert torch.equal(_ibits(nhwc_rows(o["out"].t, inp))[own], full_dx[own]), "rows scatter: own rows"
    assert o["out"].guards_ok()
    _report()


@pytest.mark.gpu
def test_device_count_zero_and_host_count_zero(dev):
    """A device count of 0 writes nothing (0 rows pad to 0 rows); a host count of 0 is refused by
    mscs_gather_normalize and writes nothing in the batched entry points."""
    from mscs_b200 import _lib as L
    lib = L.load()
    inp = make_inputs(33, 2, 48, "f16", "n=40", 77)
    d = Dev(inp, dev)
    zero = torch.zeros(1, dtype=torch.int32, device=dev)
    slot_empty = Guarded((inp.n * inp.plane,), torch.int32, dev,
                         torch.full((inp.n * inp.plane,), -1, dtype=torch.int32))
    up = 300
    o = gather_outputs(inp, dev, up)
    items = (L.GatherItem * 1)()
    gather_item(items[0], d.map.ptr(), slot_empty.ptr(), zero.data_ptr(), o, inp.n, inp.C, inp.plane, 2)
    _call(lib.mscs_gather_normalize_sectors_batch(items, 1, _stream()), "sectors gather, count 0")
    ri = (L.RowsItem * 1)()
    o2 = gather_outputs(inp, dev, up)
    rows_item(ri[0], d.nhwc.ptr(), d.pix.ptr(), zero.data_ptr(), up, inp.C, o2, 2)
    _call(lib.mscs_gather_rows_nhwc_batch(ri, 1, _stream()), "rows gather, count 0")
    torch.cuda.synchronize()
    for oo in (o, o2):
        for k in oo:
            assert bool((oo[k].buf == 0xFF).all()), f"device count 0: {k} written"
    # scatters with a device count of 0 and an upper bound: dF untouched, dense output all zeros
    for h in (False, True):
        dF = dF_dev(inp, dev, up)
        before = dF.buf.clone()
        out = Guarded((inp.n, inp.C, inp.plane), torch.float16 if h else torch.float32, dev)
        items = (L.ScatterItem * 1)()
        scatter_item(items[0], dF.ptr(), inp.ldF, o["f32"].ptr(), o["inv"].ptr(), slot_empty.ptr(), inp.n, inp.C,
                     inp.plane, out.ptr(), 2 if h else 0, zero.data_ptr())
        _call(lib.mscs_scatter_dense_batch(items, (C.c_int32 * 1)(up), 1, _stream()), "dense, count 0")
        torch.cuda.synchronize()
        assert torch.equal(dF.buf, before), "count 0: dF rows rewritten"
        assert bool((_ibits(out.t) == 0).all()) and out.guards_ok()
        ri = (L.RowsItem * 1)()
        out = Guarded((inp.n, inp.plane, inp.C), torch.float16 if h else torch.float32, dev)
        rows_item(ri[0], None, d.pix.ptr(), zero.data_ptr(), up, inp.C, o, 2 if h else 0, dF.ptr(), inp.ldF, out.ptr())
        _call(lib.mscs_scatter_rows_nhwc_batch(ri, 1, _stream()), "rows scatter, count 0")
        torch.cuda.synchronize()
        assert bool((out.buf == 0xFF).all())
    # host counts of 0
    o = gather_outputs(inp, dev, 1)
    rc = lib.mscs_gather_normalize(d.map32.ptr(), inp.n, inp.C, inp.plane, d.pix.ptr(), 0, o["bf16"].ptr(),
                                   o["f32"].ptr(), o["inv"].ptr(), None)
    assert rc < 0, "mscs_gather_normalize accepted N = 0"
    ri = (L.RowsItem * 1)()
    rows_item(ri[0], d.nhwc.ptr(), d.pix.ptr(), None, 0, inp.C, o, 2)
    _call(lib.mscs_gather_rows_nhwc_batch(ri, 1, _stream()), "rows gather, 0 rows")
    _call(lib.mscs_gather_raw_rows_batch(ri, 1, _stream()), "raw rows gather, 0 rows")
    _call(lib.mscs_gather_rows_p2p(d.nhwc.ptr(), inp.C, d.pix.ptr(), 0, None, L.ptr_array([o["bf16"].ptr()]), 1, 0, 0,
                                   o["f32"].ptr(), o["inv"].ptr(), _stream(), 2), "rows p2p, 0 rows")
    dF = dF_dev(inp, dev)
    out = Guarded((inp.n, inp.plane, inp.C), torch.float16, dev)
    rows_item(ri[0], None, d.pix.ptr(), None, 0, inp.C, o, 2, dF.ptr(), inp.ldF, out.ptr())
    _call(lib.mscs_scatter_rows_nhwc_batch(ri, 1, _stream()), "rows scatter, 0 rows")
    _call(lib.mscs_scatter_rows_pull(L.ptr_array([dF.ptr()]), 1, 0, 128, inp.ldF, o["f32"].ptr(), o["inv"].ptr(),
                                     d.pix.ptr(), 0, inp.C, out.ptr(), _stream(), 2), "rows pull, 0 rows")
    dense_out = Guarded((inp.n, inp.C, inp.plane), torch.float32, dev)
    items = (L.ScatterItem * 1)()
    scatter_item(items[0], dF.ptr(), inp.ldF, o["f32"].ptr(), o["inv"].ptr(), slot_empty.ptr(), inp.n, inp.C,
                 inp.plane, dense_out.ptr(), 0)
    before = dF.buf.clone()
    _call(lib.mscs_scatter_dense_batch(items, (C.c_int32 * 1)(0), 1, _stream()), "dense, 0 rows")
    torch.cuda.synchronize()
    for k in o:
        assert bool((o[k].buf == 0xFF).all()), f"0 rows: {k} written"
    assert bool((out.buf == 0xFF).all()), "0 rows: scatter output written"
    assert torch.equal(dF.buf, before) and bool((_ibits(dense_out.t) == 0).all())


# ---------------------------------------------------------------------------------------------------------------------
# eight items in one call: different C, plane, n and dtype, interleaved types, raw and normalised scatter items
# ---------------------------------------------------------------------------------------------------------------------
BATCH = [(256, 2, 64, "bf16", "p18"), (1, 5, 8, "f32", "all"), (200, 1, 24, "f16", "ends"),
         (33, 2, 8, "bf16", "lone7"), (128, 1, 8192, "f32", "p18"), (7, 5, 24, "f16", "octets"),
         (65, 2, 40, "f32", "lone0"), (255, 1, 16, "bf16", "all")]


@pytest.mark.gpu
def test_eight_items_match_the_single_calls(dev):
    """MSCS_MAX_SCALES items in one call, fp32 / bf16 / fp16 interleaved (the per-dtype compaction of
    gather_sectors_launch, rows_launch and dense_stream_launch), one empty item (no sampled pixel), and in the dense and
    channels-last scatters raw and normalised items mixed.  Every output equals the single-item call bit for bit."""
    from mscs_b200 import _lib as L
    lib = L.load()
    inps = [make_inputs(c, n, p, dt, ps, 900 + i, c + 5 * (i % 2)) for i, (c, n, p, dt, ps) in enumerate(BATCH)]
    # item 6: empty (no sampled pixel)
    e = inps[6]
    inps[6] = make_inputs(e.C, e.n, e.plane, e.dt, "n=0", 906, e.ldF)
    ds = [Dev(i, dev) for i in inps]
    S = len(ds)
    for kind in ("sectors", "rows", "raw", "raw_rows"):
        outs, items = [], (L.GatherItem * S)() if kind in ("sectors", "raw") else (L.RowsItem * S)()
        for s, d in enumerate(ds):
            i = d.inp
            dtc = DTYPES[i.dt][1]
            o = gather_outputs(i, dev) if kind in ("sectors", "rows") else dict(f32=Guarded((max(i.N, 1), i.C),
                                                                                              torch.float32, dev))
            if kind in ("sectors", "raw"):
                gather_item(items[s], d.map.ptr(), d.slot.ptr(), d.cnt.data_ptr(), o, i.n, i.C, i.plane, dtc)
            else:
                rows_item(items[s], d.nhwc.ptr(), d.pix.ptr(), None, i.N, i.C, o, dtc)
            outs.append(o)
        fn = dict(sectors=lib.mscs_gather_normalize_sectors_batch, rows=lib.mscs_gather_rows_nhwc_batch,
                  raw=lib.mscs_gather_raw_batch, raw_rows=lib.mscs_gather_raw_rows_batch)[kind]
        _call(fn(items, S, _stream()), kind)
        for s, d in enumerate(ds):
            single = dict(sectors=lambda: run_gather_sectors(d, True), rows=lambda: run_gather_rows(d, True),
                          raw=lambda: run_gather_raw(d, True, False), raw_rows=lambda: run_gather_raw(d, True, True))
            want = single[kind]()
            for k in outs[s]:
                assert outs[s][k].guards_ok(), f"{kind} item {s}: {k} outside its buffer"
                assert torch.equal(outs[s][k].buf, want[k].buf), f"{kind} item {s} ({d.inp.dt}, C={d.inp.C}): {k}"
            if kind == "sectors" and d.inp.N:
                check_gather_outputs("batched sectors", outs[s], d.inp)
    # scatters: even items normalised, odd items raw
    gath = [run_gather_sectors(d, True) for d in ds]
    for kind in ("dense", "rows"):
        items = (L.ScatterItem * S)() if kind == "dense" else (L.RowsItem * S)()
        outs = []
        for s, d in enumerate(ds):
            i, raw = d.inp, s % 2 == 1
            dF = dF_dev(i, dev)
            f32, inv = (None, None) if raw else (gath[s]["f32"], gath[s]["inv"])
            if kind == "dense":
                out = Guarded((i.n, i.C, i.plane), DTYPES[i.dt][0], dev)
                scatter_item(items[s], dF.ptr(), i.ldF, f32 and f32.ptr(), inv and inv.ptr(), d.slot.ptr(), i.n, i.C,
                             i.plane, out.ptr(), DTYPES[i.dt][1])
            else:
                out = Guarded((i.n, i.plane, i.C), DTYPES[i.dt][0], dev)
                rows_item(items[s], None, d.pix.ptr(), None, i.N, i.C, None if raw else dict(f32=f32, inv=inv),
                          DTYPES[i.dt][1], dF.ptr(), i.ldF, out.ptr())
            outs.append(dict(out=out, dF=dF))
        if kind == "dense":
            _call(lib.mscs_scatter_dense_batch(items, (C.c_int32 * S)(*[d.inp.N for d in ds]), S, _stream()), kind)
        else:
            _call(lib.mscs_scatter_rows_nhwc_batch(items, S, _stream()), kind)
        for s, d in enumerate(ds):
            raw = s % 2 == 1
            f32, inv = gath[s]["f32"], gath[s]["inv"]
            want = (run_scatter_dense if kind == "dense" else run_scatter_rows)(d, f32, inv, True, raw=raw)
            for k in ("out", "dF"):
                assert outs[s][k].guards_ok()
                assert torch.equal(outs[s][k].buf, want[k].buf), f"{kind} item {s} ({d.inp.dt}, raw={raw}): {k}"
    _report()


# ---------------------------------------------------------------------------------------------------------------------
# pooled: worlds 1, 2, 3, 8 on one GPU, every slab an ordinary device buffer
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("dt", ["f32", "bf16", "f16"])
def test_pooled_entry_points(world, dt, dev):
    """Rank r owns images [r n_l, (r+1) n_l) of one global map; rows are in a random (global) order; gradient rows are
    sharded in blocks of rows_per_rank = 128 rows, the last rank short.  After each rank's p2p gather, the rows of the
    other ranks are untouched in every slab and only the own slab's padding rows are zeroed; after all ranks every slab
    holds the same rows.  The pull scatters of every rank equal the single-process scatter bit for bit."""
    from mscs_b200 import _lib as L
    n_l, plane, Cc, rpr = 2, 96, 129 if dt == "f32" else 63, 128
    N = rpr * (world - 1) + 70
    inp = make_inputs(Cc, n_l * world, plane, dt, f"n={N}", 31 * world + len(dt), Cc + 4)
    d = Dev(inp, dev)
    owner = (inp.pix // plane) // n_l                        # rank whose images hold the row's pixel
    local = n_l * plane
    esz = torch.empty((), dtype=DTYPES[dt][0]).element_size()
    single = run_gather_rows(d, True)
    single_p2p = run_gather_p2p(d, True)
    for layout in ("nchw", "nhwc"):
        nb = inp.N_pad * inp.C_pad * 2
        slabs = p2p_slabs(world, nb, P2P_OFF, dev)
        o = gather_outputs(inp, dev)
        for r in range(world):
            pix_r = torch.from_numpy(np.where(owner == r, inp.pix - r * local, -1).astype(np.int32)).to(dev)
            if layout == "nhwc":
                run_gather_rows_p2p(d, True, world, r, slabs, pix=pix_r.data_ptr(),
                                    feat=d.nhwc.ptr() + r * local * Cc * esz, o=o)
            else:
                run_gather_p2p(d, True, world, r, slabs, slot=d.slot.ptr() + r * local * 4,
                               feat=d.map.ptr() + r * local * Cc * esz, n=n_l, o=o)
            torch.cuda.synchronize()
            done = torch.from_numpy(owner <= r)
            for q, s in enumerate(slabs):
                m = _host(slab_view(s, P2P_OFF, (inp.N_pad, inp.C_pad), torch.int16))
                assert bool((m[:N][~done] == -1).all()), f"rank {r} wrote rows of other ranks into slab {q}"
                pad_zero = bool((m[N:] == 0).all())
                assert pad_zero == (q <= r) or N == inp.N_pad, f"rank {r}: padding rows of slab {q}"
                assert s.guards_ok()
        ref = single if layout == "nhwc" else single_p2p
        for q, s in enumerate(slabs):
            m = _host(slab_view(s, P2P_OFF, (inp.N_pad, inp.C_pad), torch.int16))
            want = _host(ref["bf16"].bits()) if layout == "nhwc" else _host(
                slab_view(ref["slab0"], P2P_OFF, (inp.N_pad, inp.C_pad), torch.int16))
            assert torch.equal(m, want), f"{layout}: slab {q} differs from the single-process rows"
        assert torch.equal(_host(o["f32"].bits()), _host(ref["f32"].bits())), f"{layout}: fp32 rows"
        assert torch.equal(_host(o["inv"].bits()), _host(ref["inv"].bits())), f"{layout}: inv_norm"
        if layout == "nchw":
            check_gather_outputs("k_gather_p2p pooled", dict(f32=o["f32"], inv=o["inv"]), inp)
    # pull scatters: each rank scatters its own images, reading row i from slab i // rpr
    f32, inv = single["f32"], single["inv"]
    want_rows = run_scatter_rows(d, f32, inv, True)["out"]
    want_grad = run_scatter_grad(d, f32, inv, 0)["out"]
    slabs = pull_slabs(inp, world, rpr, dev)
    for layout in ("nchw", "nhwc"):
        for r in range(world):
            pix_r = torch.from_numpy(np.where(owner == r, inp.pix - r * local, -1).astype(np.int32)).to(dev)
            o = run_pull(d, f32, inv, True, layout == "nhwc", world, rpr, slabs, slot=d.slot.ptr() + r * local * 4,
                         pix=pix_r.data_ptr(), n=n_l)
            assert o["out"].guards_ok()
            if layout == "nhwc":
                want = _host(want_rows.t[r * n_l:(r + 1) * n_l])
                assert torch.equal(_ibits(_host(o["out"].t)), _ibits(want)), f"rows pull rank {r}"
            else:
                want = _host(want_grad.t[r * n_l:(r + 1) * n_l]).to(DTYPES[dt][0])
                got = _host(o["out"].t)
                m = torch.from_numpy(sampled_mask(inp)[r * n_l:(r + 1) * n_l])[:, None, :].expand_as(got)
                assert torch.equal(_ibits(got)[m], _ibits(want)[m]), f"sectors pull rank {r}"
                om = torch.from_numpy(octet_mask(inp)[r * n_l:(r + 1) * n_l])[:, None, :].expand_as(got)
                assert bool((_ibits(got)[~om] == -1).all()) and bool((_ibits(got)[om & ~m] == 0).all())
    _report()


# ---------------------------------------------------------------------------------------------------------------------
# element offsets above 2^31
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_element_offsets_above_2_to_the_31(dev):
    """A bf16 NCHW map with n C plane = 40 x 256 x (480 x 512) = 2.5e9 elements (2^31 < 2.5e9 < 2^32): the sector
    gather, the dense writer and the bf16 pull scatter at world 1, with sampled pixels in the first and the last images.
    Checked on the device (indexing, count_nonzero); nothing of the 5 GB buffers is copied to the host."""
    from mscs_b200 import _lib as L
    lib = L.load()
    n, Cc, plane = 40, 256, 480 * 512
    assert (1 << 31) < n * Cc * plane < (1 << 32)
    rs = np.random.RandomState(2024)
    imgs = np.array([0, 1, 37, 38, 39, 39, 39])
    pix = np.unique(imgs * plane + rs.randint(0, plane, len(imgs)))
    pix = np.concatenate([pix, [n * plane - 1, (n - 1) * plane]])
    pix = rs.permutation(np.unique(pix)).astype(np.int32)
    N = len(pix)
    vals = torch.from_numpy(rs.standard_normal((N, Cc))).to(torch.bfloat16)
    feat = torch.full((n, Cc, plane), float("nan"), dtype=torch.bfloat16, device=dev)
    bi, pi = torch.from_numpy(pix // plane).long().to(dev), torch.from_numpy(pix % plane).long().to(dev)
    feat[bi, :, pi] = vals.to(dev)
    slot = torch.full((n * plane,), -1, dtype=torch.int32, device=dev)
    slot[torch.from_numpy(pix).long().to(dev)] = torch.arange(N, dtype=torch.int32, device=dev)
    cnt = torch.tensor([N], dtype=torch.int32, device=dev)
    inp = types.SimpleNamespace(C=Cc, N=N, C_pad=256, N_pad=256, x64=vals.double().numpy())
    o = gather_outputs(inp, dev)
    items = (L.GatherItem * 1)()
    gather_item(items[0], feat.data_ptr(), slot.data_ptr(), cnt.data_ptr(), o, n, Cc, plane, 1)
    _call(lib.mscs_gather_normalize_sectors_batch(items, 1, _stream()), "sectors gather")
    f, iv, _ = check_gather_outputs("sectors gather above 2^31", o, inp)
    g = torch.from_numpy(rs.standard_normal((N, Cc)).astype(np.float32))
    dF = g.to(dev).clone()
    out = torch.full((n, Cc, plane), float("nan"), dtype=torch.bfloat16, device=dev)
    items = (L.ScatterItem * 1)()
    scatter_item(items[0], dF.data_ptr(), Cc, o["f32"].ptr(), o["inv"].ptr(), slot.data_ptr(), n, Cc, plane,
                 out.data_ptr(), 1)
    _call(lib.mscs_scatter_dense_batch(items, (C.c_int32 * 1)(N), 1, _stream()), "dense writer")
    dx = dF.cpu()                                             # k_dx_rows: dx in place
    fails, w = check_dx(f, iv, g.numpy(), dx.numpy())
    _worst("k_dx_rows above 2^31", w)
    assert not fails, fails
    want = dx.to(torch.bfloat16)
    got = out[bi, :, pi].cpu()
    assert torch.equal(_ibits(got), _ibits(want)), "dense writer: sampled pixels"
    assert int(torch.count_nonzero(out)) == int(torch.count_nonzero(want)), "dense writer: non-zero (or NaN) elsewhere"
    out.fill_(float("nan"))
    slab = torch.full((P2P_OFF // 4 + N * Cc,), float("nan"), dtype=torch.float32, device=dev)
    slab[P2P_OFF // 4:] = g.to(dev).ravel()
    _call(lib.mscs_scatter_sectors_pull(L.ptr_array([slab.data_ptr()]), 1, P2P_OFF, 128, Cc, o["f32"].ptr(),
                                        o["inv"].ptr(), slot.data_ptr(), n, Cc, plane, out.data_ptr(), _stream(), 1),
          "bf16 pull scatter")
    got = out[bi, :, pi].cpu()
    assert torch.equal(_ibits(got), _ibits(want)), "pull scatter: sampled pixels"
    octs = np.unique(pix // 8)
    assert int(torch.isnan(out).sum()) == n * Cc * plane - len(octs) * 8 * Cc, "pull scatter: octet extent"
    assert int(torch.count_nonzero(torch.nan_to_num(out, nan=0.0))) == int(torch.count_nonzero(want))
    del feat, out, slot
    torch.cuda.empty_cache()
    _report()
