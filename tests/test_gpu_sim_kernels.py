"""The tensor-core similarity kernels (K3 ``k_sim_fwd`` / K4 ``k_sim_bwd``) driven directly through the C ABI, without
sampling or gather in front, against the fp64 oracle evaluated on the SAME bf16 operand rows.

Every channel-width instance (C_pad / 64 = KB = 1..4), row counts at and one off the 32-row warp groups, 128-row tiles
and 256-key blocks, class layouts from one class to a boundary in every warp, and clustered embeddings (the regime a
model in training produces: positive logits near 1/tau, u = e_ij / neg_i from 1/64 to >> 1, hard negatives) are
compared row by row.  The device-count instances, row ranges and set masks are compared with the plain call.

Error model (see ``compare``).  With the oracle on the bf16 rows widened to fp64, what is left is accumulation order,
the ex2 / lg2 / rcp approximations, fp32 evaluation and the bf16 rounding of W in the backward:

* row statistics neg_i, pos_i, S_i: the fp32 torch port of the reference (oracle/torch_port.py, same rows) makes the
  same kind of fp32 errors -- including the cancellation in pos_i = sum [l_ij - log(e_ij + neg_i)] when e_ij >> neg_i --
  so its distance from fp64 is the budget:  |k_i - o_i| <= A_STATS * (|port_i - o_i| + eps32 * K_i),  where K_i is the
  first-order fp32 condition sum of the row (sum_neg e(1+|l|) for neg_i; for pos_i and S_i the same with the error of
  den = e + neg_i carried through log / reciprocal).  eps32 * K_i is one fp32 ulp of the row's terms: a floor for rows
  where the port happens to land on the fp64 value.
* term losses and the total: the same bound on the mean, or the 1e-3 relative north-star bound where that is looser.
* dF (d loss / d unit rows): the kernel rounds W to bf16 before dX += W Y, with W from fp32 coefficients.  The fp32
  value of W differs from the fp64 one by ~1e-6 relative, so it rounds to the SAME bf16 value except next to a rounding
  boundary: emulating the rounding on the fp64 W (``_reference``: W as in the header of sim_bwd.cu, through fp32 to
  bf16, times the fp64 rows) reproduces the kernel's error row by row.  Bound:
  ||dF_i - dF64_i|| <= A_DF * (||emul_i - dF64_i|| + eps32 * sum_j |W_ij| ||Y_j|| * |scale|),  the second term being
  the fp32 accumulation of the tensor-core product; then max-abs and a global cosine as a second line.

A_STATS and A_DF were calibrated on an NVIDIA B200 (worst observed ratios next to them below and in DESIGN.md §2).
``test_comparator_*`` (no GPU) shows that these bounds reject simulated kernel faults and accept the emulation.
"""
import ctypes as C
import math
import types

import numpy as np
import pytest
import torch

from helpers import cosine

EPS32 = 2.0 ** -23            # fp32 ulp of 1
# Calibrated on an NVIDIA B200 (1000 W power limit): worst observed ratio 3.52 for the row statistics (c256_n1500_hard),
# 2.90 for dF (c192_n1500_edges_det3) over every case, device-count, row-range and set-mask run; the simulated faults
# of test_comparator_rejects_simulated_kernel_faults reach 33 and more.
A_STATS = 8.0                 # row statistics / losses: kernel error <= A_STATS x (fp32 port error + 1 ulp floor)
A_DF = 8.0                    # dF rows: kernel error <= A_DF x (bf16-W emulation error + fp32 accumulation floor)
NORTH_STAR_REL = 1e-3         # loss bound of BASELINE.json, used where it is looser
NUM_CLASSES = 200
U_SERIES = 1.0 / 64           # k_sim_fwd: the positive sweep takes the series path while e * (1 / neg_i) < 1/64


# ---------------------------------------------------------------------------------------------------------------------
# inputs: class layouts and geometries
# ---------------------------------------------------------------------------------------------------------------------
def _edge_sizes(N):
    """class boundaries exactly at and one past multiples of 32 / 128 / 256 (alternating), every class >= 2 rows."""
    bounds = []
    for k in range(1, N // 32 + 1):
        off = (k % 2) if k % 4 else (k // 4) % 2      # 33, 64, 97, 128, 161, 192, 225, 257, 289, 320, ..., 384, ..., 513
        b = 32 * k + off
        if 2 <= b <= N - 2:
            bounds.append(b)
    edges = [0] + bounds + [N]
    return [b - a for a, b in zip(edges[:-1], edges[1:])]


def class_layout(kind, N, rs, pool):
    """Sorted class ids (N,) drawn from ``pool``; every class has >= 2 rows (a single-row class of a self term is 0/0 in
    the reference too, and the sampler never produces one)."""
    assert N >= 2
    if kind == "one" or N < 4:
        sizes = [N]
    elif kind == "two":
        sizes = [N // 2, N - N // 2]
    elif kind == "ade":        # ADE20K-like: many classes of 2..~12 rows, a class boundary in almost every warp
        k = int(min(len(pool), max(2, N // 7)))
        sizes = list(2 + rs.multinomial(N - 2 * k, rs.dirichlet(np.ones(k))))
    elif kind == "big":        # one class of ~600 rows across several 128-row tiles, small classes around it
        big = min(600, N - 40)
        rest = N - big
        k = int(min(len(pool) - 1, max(2, rest // 7)))
        sizes = list(2 + rs.multinomial(rest - 2 * k, rs.dirichlet(np.ones(k))))
        sizes.insert(len(sizes) // 3, big)
    elif kind == "edges":
        sizes = _edge_sizes(N)
    else:
        raise ValueError(kind)
    assert sum(sizes) == N and min(sizes) >= 2 and len(sizes) <= len(pool)
    ids = np.sort(rs.choice(pool, len(sizes), replace=False))
    return np.repeat(ids, sizes).astype(np.int64)


def centroids(C, geom, rs):
    """one unit centroid per class; "hard": class 2k+1 sits next to class 2k (cosine ~0.92): hard negatives."""
    mu = rs.standard_normal((NUM_CLASSES, C))
    mu /= np.linalg.norm(mu, axis=1, keepdims=True)
    if geom == "hard":
        h = rs.standard_normal((NUM_CLASSES // 2, C))
        h /= np.linalg.norm(h, axis=1, keepdims=True)
        mu[1::2] = mu[0::2] + 0.42 * h
        mu[1::2] /= np.linalg.norm(mu[1::2], axis=1, keepdims=True)
    return mu


def _unit(x):
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def bf16_round(x):
    """fp64 -> fp32 -> bf16 (round to nearest even, as the kernels and the gather store) -> fp64."""
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).double().numpy()


def positive_u(F, y, tau, max_rows=None):
    """u_ij = e_ij / neg_i of every positive pair of the self term on rows F (fp64), and the row of each pair;
    rows without negatives are skipped."""
    N = F.shape[0] if max_rows is None else min(F.shape[0], max_rows)
    us, rows = [], []
    for r0 in range(0, N, 512):
        r1 = min(N, r0 + 512)
        E = np.exp(F[r0:r1] @ F.T / tau)
        same = y[r0:r1, None] == y[None, :]
        neg = (E * ~same).sum(1)
        same[np.arange(r1 - r0), np.arange(r0, r1)] = False
        ok = neg > 0
        ri, cj = np.nonzero(same & ok[:, None])
        us.append(E[ri, cj] / neg[ri])
        rows.append(ri + r0)
    return np.concatenate(us), np.concatenate(rows)


# target median u of the positives of set 0 per clustered geometry (the spread sigma is found by bisection)
U_TARGET = {"straddle": U_SERIES, "converged": 100.0, "hard": 0.5}


def _clustered(mu, cls, sigma, noise):
    return _unit(mu[cls] + sigma * noise)


def make_rows(geom, cls_list, C, tau, rs):
    """fp64 unit rows per set.  "iid": Gaussian noise (nearly orthogonal rows, logits ~0, u ~ 1/N); clustered:
    normalize(mu_c + sigma g) with sigma chosen so that the median u of the positives of set 0 hits U_TARGET[geom]."""
    noise = [rs.standard_normal((len(c), C)) / math.sqrt(C) for c in cls_list]
    if geom == "iid":
        return [_unit(n) for n in noise]
    mu = centroids(C, geom, rs)
    lo, hi = math.log(0.02), math.log(20.0)       # median u falls as sigma grows
    for _ in range(24):
        mid = 0.5 * (lo + hi)
        u, _ = positive_u(_clustered(mu, cls_list[0], math.exp(mid), noise[0]), cls_list[0], tau, max_rows=384)
        if np.median(u) > U_TARGET[geom]:
            lo = mid
        else:
            hi = mid
    sigma = math.exp(0.5 * (lo + hi))
    return [_clustered(mu, c, sigma, n) for c, n in zip(cls_list, noise)]


def check_regime(geom, F, y, tau):
    """The clustered cases assert the regime they claim, so that a change to the generator cannot drop the coverage.
    Returns (share of positive pairs with u >= 1/64, description)."""
    u, rows = positive_u(F, y, tau)
    if len(u) == 0:
        return float("nan"), "no positive pairs with negatives"
    share = float(np.mean(u >= U_SERIES))
    if geom == "straddle":
        assert 0.05 <= share <= 0.95, f"straddling case: share of u >= 1/64 is {share:.3f}"
        g = rows // 32
        hi = np.bincount(g, weights=(u >= U_SERIES), minlength=g.max() + 1)
        tot = np.bincount(g, minlength=g.max() + 1)
        assert np.any((hi > 0) & (hi < tot)), "no 32-row group mixes the series and the lg2/rcp path"
    elif geom == "converged":
        assert np.mean(u >= 10.0) >= 0.75, f"converged case: only {np.mean(u >= 10.0):.3f} of the pairs have u >= 10"
    elif geom == "hard":
        # the twin class (centroid next to this one) carries most of neg_i for most rows that have it
        E = np.exp(F @ F.T / tau)
        twin = (y[None, :] == (y[:, None] ^ 1))
        neg = (E * (y[:, None] != y[None, :])).sum(1)
        has = twin.any(1)
        share_twin = (E * twin).sum(1)[has] / neg[has]
        assert has.mean() > 0.3 and np.mean(share_twin > 0.5) >= 0.5, "hard-negative case: twins do not dominate neg_i"
    return share, f"u median {np.median(u):.3g}"


# ---------------------------------------------------------------------------------------------------------------------
# the case matrix
# ---------------------------------------------------------------------------------------------------------------------
# id: (C, rows per set, class layout, geometry, temperature, terms, grad_out)
#   terms: self = single-scale terms only; ms_cs = 2 scales + cross-scale; ms3 = 3 scales (w_high_mid term);
#          detach = detach_deepest (no key-side pass); eight = 8 sets (10 terms);
#          mismatch = cross-scale whose anchor / key sets have classes the other side lacks
CASES = {
    "c8_n2_one":            (8,   [2], "one", "iid", 0.1, "self", 0.7),
    "c8_n31_two":           (8,   [31], "two", "iid", 0.5, "self", -2.5),
    "c8_n513_edges":        (8,   [513], "edges", "iid", 0.1, "self", 0.7),
    "c64_n32_ade":          (64,  [32], "ade", "iid", 0.07, "self", 0.7),
    "c64_n127_edges":       (64,  [127], "edges", "straddle", 0.07, "self", 0.7),
    "c64_n128_two_cs":      (64,  [128, 33], "two", "iid", 0.1, "ms_cs", 0.7),
    "c64_n129_ade":         (64,  [129], "ade", "converged", 0.07, "self", -2.5),
    "c64_n1500_ade":        (64,  [1500], "ade", "converged", 0.07, "self", 0.7),
    "c64_eight":            (64,  [130, 64, 40, 33, 32, 31, 12, 2], "ade", "iid", 0.1, "eight", 0.0),
    "c100_n255_ade_cs":     (100, [255, 64], "ade", "straddle", 0.07, "ms_cs", 0.7),
    "c100_n256_edges":      (100, [256], "edges", "iid", 0.5, "self", 0.0),
    "c128_n257_two":        (128, [257], "two", "converged", 0.1, "self", 0.7),
    "c128_n383_ade_ms3":    (128, [383, 129, 40], "ade", "straddle", 0.07, "ms3", 0.7),
    "c128_n513_hard":       (128, [513], "ade", "hard", 0.07, "self", -2.5),
    "c150_n2_one":          (150, [2], "one", "iid", 0.07, "self", 0.7),
    "c150_n31_two_cs":      (150, [31, 2], "two", "iid", 0.1, "ms_cs", -2.5),
    "c150_n32_ade":         (150, [32], "ade", "straddle", 0.07, "self", 0.7),
    "c150_n127_ade":        (150, [127], "ade", "straddle", 0.07, "self", 0.7),
    "c150_n128_two":        (150, [128], "two", "converged", 0.07, "self", -2.5),
    "c150_n129_edges_det":  (150, [129, 257], "edges", "iid", 0.1, "detach", 0.7),
    "c150_n255_hard":       (150, [255], "ade", "hard", 0.07, "self", 0.7),
    "c150_n256_edges_ms3":  (150, [256, 128, 31], "edges", "straddle", 0.07, "ms3", 0.7),
    "c150_n257_mismatch":   (150, [257, 200], "ade", "converged", 0.07, "mismatch", 0.7),
    "c150_n383_ade":        (150, [383], "ade", "iid", 0.5, "self", 0.0),
    "c150_n513_edges":      (150, [513], "edges", "straddle", 0.07, "self", -2.5),
    "c150_n1500_big_cs":    (150, [1500, 383], "big", "straddle", 0.07, "ms_cs", 0.7),
    "c192_n257_one":        (192, [257], "one", "iid", 0.1, "self", 0.7),
    "c192_n1500_big":       (192, [1500], "big", "converged", 0.1, "self", 0.7),
    "c192_n1500_edges_det3": (192, [1500, 513, 129], "edges", "hard", 0.07, "detach", -2.5),
    "c192_n4000_ade":       (192, [4000], "ade", "straddle", 0.07, "self", 0.7),
    "c200_n383_edges_ms3":  (200, [383, 255, 127], "edges", "iid", 0.1, "ms3", 0.7),
    "c200_n129_mismatch":   (200, [129, 255], "ade", "converged", 0.07, "mismatch", -2.5),
    "c256_n128_ade":        (256, [128], "ade", "iid", 0.1, "self", 0.7),
    "c256_n129_edges":      (256, [129], "edges", "straddle", 0.07, "self", 0.7),
    "c256_n256_two":        (256, [256], "two", "converged", 0.07, "self", 0.0),
    "c256_n257_edges_ms3":  (256, [257, 256, 129], "edges", "straddle", 0.07, "ms3", -2.5),
    "c256_n513_mismatch":   (256, [513, 383], "ade", "iid", 0.5, "mismatch", 0.7),
    "c256_n1500_hard":      (256, [1500], "ade", "hard", 0.07, "self", -2.5),
    "c256_n4000_big_cs":    (256, [4000, 1500], "big", "converged", 0.07, "ms_cs", 0.7),
    "c256_eight":           (256, [383, 257, 129, 128, 127, 33, 32, 31], "edges", "straddle", 0.07, "eight", 0.7),
}


def make_spec(terms, S, tau):
    from mscs_b200 import _ops
    cs = terms != "self"
    weights = [1.0, 0.7, 0.4, 0.1, 0.3, 0.2, 0.6, 0.5][:S]
    return _ops.LossSpec(num_classes=NUM_CLASSES, temperature=tau, cs_temperature=0.1 if tau == 0.07 else tau,
                         weights=weights, cross_scale=cs, detach_deepest=terms == "detach",
                         w_high_low=0.8 if cs else 1.0, w_high_mid=0.6 if cs else 1.0)


def term_list(spec, S):
    """the terms of build_job, in its order: (anchor set, key set, self term, weight, tau, key-side pass)."""
    terms = [(s, s, True, spec.weights[s], spec.temperature, False) for s in range(S)]
    if spec.cross_scale:
        terms.append((0, S - 1, False, spec.w_high_low, spec.cs_temperature, not spec.detach_deepest))
        if S > 2:
            terms.append((0, S - 2, False, spec.w_high_mid, spec.cs_temperature, not spec.detach_deepest))
    return terms


def make_case(name):
    C_, Ns, layout, geom, tau, terms, g = CASES[name]
    rs = np.random.RandomState(sum(map(ord, name)) * 7919 % (1 << 31))      # fixed per case name
    S = len(Ns)
    pools = [np.arange(NUM_CLASSES)] * S
    if terms == "mismatch":      # anchors: classes 0..119, keys: 40..199 -> classes on one side only, both ways
        pools = [np.arange(0, 120)] + [np.arange(40, NUM_CLASSES)] * (S - 1)
    cls = [class_layout(layout if N >= 4 else "one", N, rs, p) for N, p in zip(Ns, pools)]
    if geom == "hard":           # twins: classes 2k and 2k+1 next to each other in the layout
        cls = [_pair_twins(c, rs) for c in cls]
    F = make_rows(geom, cls, C_, tau, rs)
    rows = [bf16_round(f) for f in F]           # the operand rows the kernels read, widened exactly to fp64
    spec = make_spec(terms, S, tau)
    return types.SimpleNamespace(name=name, C=C_, KB=(C_ + 63) // 64, Ns=Ns, layout=layout, geom=geom, tau=tau,
                                 terms=terms, g=g, cls=cls, rows=rows, spec=spec, S=S)


def _pair_twins(c, rs):
    """map each run of classes onto twin pairs (2k, 2k+1) so hard negatives sit next to their class."""
    ids = np.unique(c)
    new = np.empty_like(ids)
    base = np.sort(rs.choice(NUM_CLASSES // 2, (len(ids) + 1) // 2, replace=False)) * 2
    for i in range(len(ids)):
        new[i] = base[i // 2] + (i % 2)
    return new[np.searchsorted(ids, c)]


# ---------------------------------------------------------------------------------------------------------------------
# reference: fp64 oracle, fp32 port, bf16-W emulation and the error-model sums
# ---------------------------------------------------------------------------------------------------------------------
def _port_stats(Fa, ya, Fk, yk, tau, self_mask):
    """fp32 torch port (oracle/torch_port.py) on the same rows: its loss, and the per-row statistics computed with the
    same ops (exp of the fp32 logits, masked sums, log(e + neg))."""
    from oracle import torch_port
    a, k = torch.from_numpy(Fa).float(), torch.from_numpy(Fk).float()
    logits = torch.matmul(a, k.t()) / tau
    same = torch.from_numpy(ya[:, None] == yk[None, :]).float()
    pos = same.clone()
    if self_mask:
        pos.fill_diagonal_(0.0)
    neg = 1 - same
    loss = float(torch_port._masked_nll(logits, pos, neg, guard=not self_mask))
    e = torch.exp(logits)
    neg_sum = (e * neg).sum(1, keepdim=True)
    den = e + neg_sum
    possum = (pos * (logits - torch.log(den))).sum(1)
    S = (pos / den).sum(1)
    return dict(neg=neg_sum[:, 0].double().numpy(), possum=possum.double().numpy(), S=S.double().numpy(), loss=loss)


def _reference(case, chunk=512):
    from oracle import loss_fp64
    rows, ys, S = case.rows, case.cls, case.S
    g = case.g
    terms = term_list(case.spec, S)
    out = types.SimpleNamespace(terms=[], total=0.0, total_K=0.0)
    dF64 = [np.zeros_like(r) for r in rows]
    emul = [np.zeros_like(r) for r in rows]
    mine = [np.zeros_like(r) for r in rows]
    absW = [np.zeros(len(r)) for r in rows]
    ynorm = [np.linalg.norm(r, axis=1) for r in rows]
    for (a, k, self_mask, w, tau, need_dk) in terms:
        Fa, Fk, ya, yk = rows[a], rows[k], ys[a], ys[k]
        N1, N2 = len(Fa), len(Fk)
        loss, dFa, dFk, st = loss_fp64.term(Fa, ya, Fk, yk, tau, self_mask, True, 1024)
        port = _port_stats(Fa, ya, Fk, yk, tau, self_mask)
        P = st["P"]
        div = P if self_mask else np.where(P > 0, P, 1.0)
        c = 1.0 / (div * N1)
        cS, cPN, neg = st["S"] * c, st["neg"] * c, st["neg"]
        K = dict(neg=np.zeros(N1), possum=np.zeros(N1), S=np.zeros(N1))
        scale = w / tau * g
        for r0 in range(0, N1, chunk):
            r1 = min(N1, r0 + chunk)
            L = Fa[r0:r1] @ Fk.T / tau
            E = np.exp(L)
            same = ya[r0:r1, None] == yk[None, :]
            pos = same.copy()
            if self_mask:
                pos[np.arange(r1 - r0), np.arange(r0, r1)] = False
            n_i = neg[r0:r1, None]
            den = E + n_i
            kneg = (E * (1 + np.abs(L)) * ~same).sum(1)
            dden = E * (1 + np.abs(L)) + kneg[:, None]          # first-order fp32 error of den, in ulps
            K["neg"][r0:r1] = kneg
            K["possum"][r0:r1] = (pos * (np.abs(L) + np.abs(np.log(den)) + dden / den)).sum(1)
            K["S"][r0:r1] = (pos * (1 + dden / den) / den).sum(1)
            # W of sim_bwd.cu: row coefficients (and, for a self term, the column coefficients: W = G + G^T)
            Gr = np.where(pos, -cPN[r0:r1, None] / den, np.where(same, 0.0, E * cS[r0:r1, None]))
            if self_mask:
                Wc = np.where(pos, -cPN[None, :] / (E + neg[None, :]), np.where(same, 0.0, E * cS[None, :]))
                W = Gr + Wc
            else:
                W = Gr
            Wb = bf16_round(W)
            emul[a][r0:r1] += scale * (Wb @ Fk)
            mine[a][r0:r1] += scale * (W @ Fk)
            absW[a][r0:r1] += abs(scale) * (np.abs(W) @ ynorm[k])
            if need_dk:      # key-side pass: rows = keys, W_ji = G_ij (row coefficients of the anchors only)
                Gb = bf16_round(Gr)
                emul[k] += scale * (Gb.T @ Fa[r0:r1])
                mine[k] += scale * (Gr.T @ Fa[r0:r1])
                absW[k] += abs(scale) * (np.abs(Gr).T @ ynorm[a][r0:r1])
        dF64[a] += w * g * dFa
        if self_mask:
            dF64[a] += w * g * dFk
        elif need_dk:
            dF64[k] += w * g * dFk
        K_loss = float(np.sum(K["possum"] / div) / N1)
        out.terms.append(dict(a=a, k=k, self_mask=self_mask, w=w, N1=N1, loss=loss, st=st, div=div, port=port, K=K,
                              K_loss=K_loss))
        out.total += w * loss
        out.total_K += abs(w) * K_loss
    out.port_total = sum(t["w"] * t["port"]["loss"] for t in out.terms)
    for s in range(S):      # the emulation's W is the oracle's: same product in fp64
        np.testing.assert_allclose(mine[s], dF64[s], rtol=1e-9, atol=1e-12 * (np.abs(dF64[s]).max() + 1e-300))
    out.dF64, out.emul, out.absW = dF64, emul, absW
    return out


# ---------------------------------------------------------------------------------------------------------------------
# comparator
# ---------------------------------------------------------------------------------------------------------------------
def compare(ref, got, g):
    """``got``: kernel outputs, dict(terms=[dict(neg, possum, S, coef_s, coef_pn, loss)], total, flag, dF=[per set]).
    Returns (list of failures, dict of the worst ratio of each kind: error / (budget without the factor A))."""
    fails, worst = [], dict(stats=0.0, loss=0.0, dF=0.0)
    for ti, (rt, gt) in enumerate(zip(ref.terms, got["terms"])):
        for key in ("neg", "possum", "S"):
            o, k_, p = rt["st"][key], np.asarray(gt[key], np.float64), rt["port"][key]
            unit = np.abs(p - o) + EPS32 * rt["K"][key] + 1e-30
            r = np.abs(k_ - o) / unit
            r = np.where(np.isnan(r), np.inf, r)
            worst["stats"] = max(worst["stats"], float(r.max()))
            if r.max() > A_STATS:
                i = int(np.argmax(r))
                fails.append(f"term {ti} {key}: row {i} (tile {i // 128}, group {i // 32}) kernel {k_[i]:.9g} fp64 "
                             f"{o[i]:.9g} port {p[i]:.9g}: ratio {r[i]:.3g}")
        # the backward coefficients are the kernel's own statistics over div_i * N1
        n1d = rt["div"] * rt["N1"]
        for key, src in (("coef_s", "S"), ("coef_pn", "neg")):
            want = np.asarray(gt[src], np.float64) / n1d
            err = np.abs(np.asarray(gt[key], np.float64) - want)
            if not np.all(err <= 4 * EPS32 * np.abs(want) + 1e-38):
                i = int(np.nanargmax(np.where(np.isnan(err), np.inf, err)))
                fails.append(f"term {ti} {key}: row {i} {gt[key][i]:.9g} vs {src}/(div N1) {want[i]:.9g}")
        o, p = rt["loss"], rt["port"]["loss"]
        unit = abs(p - o) + EPS32 * rt["K_loss"]
        err = abs(float(gt["loss"]) - o)
        worst["loss"] = max(worst["loss"], err / max(unit, 1e-30))
        if not err <= max(A_STATS * unit, NORTH_STAR_REL * abs(o)):
            fails.append(f"term {ti} loss: kernel {float(gt['loss']):.9g} fp64 {o:.9g} port {p:.9g}")
    err = abs(float(got["total"]) - ref.total)
    if not err <= max(A_STATS * (abs(ref.port_total - ref.total) + EPS32 * ref.total_K), NORTH_STAR_REL * abs(ref.total)):
        fails.append(f"total: kernel {float(got['total']):.9g} fp64 {ref.total:.9g}")
    if float(got["flag"]) != 0.0:
        fails.append("inf/NaN flag set")
    for s, d in enumerate(got["dF"]):
        d = np.asarray(d, np.float64)
        d64, em = ref.dF64[s], ref.emul[s]
        if g == 0.0:
            if not np.all(d == 0.0):
                fails.append(f"set {s}: dF not exactly zero for grad_out 0")
            continue
        e_k = np.linalg.norm(d - d64, axis=1)
        unit = np.linalg.norm(em - d64, axis=1) + EPS32 * ref.absW[s] + 1e-300
        r = e_k / unit
        r = np.where(np.isnan(r), np.inf, r)
        worst["dF"] = max(worst["dF"], float(r.max()))
        if r.max() > A_DF:
            i = int(np.argmax(r))
            fails.append(f"set {s} dF: row {i} (tile {i // 128}, group {i // 32}) |err| {e_k[i]:.3e} emulated "
                         f"{np.linalg.norm(em[i] - d64[i]):.3e} |dF64| {np.linalg.norm(d64[i]):.3e}: ratio {r[i]:.3g}")
        # second line: max-abs and a global cosine
        mx = np.abs(d - d64).max()
        mx_b = A_DF * (np.abs(em - d64).max() + EPS32 * ref.absW[s].max())
        if not mx <= mx_b:
            fails.append(f"set {s} dF: max-abs {mx:.3e} > {mx_b:.3e}")
        if np.abs(d64).max() > 0:
            cs_ = cosine(d, d64)
            cs_e = cosine(em, d64)
            if not cs_ >= 1.0 - A_DF * max(1.0 - cs_e, 1e-12):
                fails.append(f"set {s} dF: cosine {cs_:.10f} (emulated {cs_e:.10f})")
    return fails, worst


def ref_as_got(ref, case):
    """what an exact kernel with the bf16-W rounding would return: fp64 statistics, the emulated dF."""
    terms = []
    for rt in ref.terms:
        st = rt["st"]
        terms.append(dict(neg=st["neg"], possum=st["possum"], S=st["S"], coef_s=st["S"] / (rt["div"] * rt["N1"]),
                          coef_pn=st["neg"] / (rt["div"] * rt["N1"]), loss=rt["loss"]))
    return dict(terms=terms, total=ref.total, flag=0.0, dF=[e.copy() for e in ref.emul])


_CACHE = {}


def case_and_ref(name):
    if name not in _CACHE:
        case = make_case(name)
        share, what = (check_regime(case.geom, case.rows[0], case.cls[0], case.tau) if case.geom != "iid"
                       else (float(np.mean(positive_u(case.rows[0], case.cls[0], case.tau)[0] >= U_SERIES))
                             if case.Ns[0] > 2 and len(np.unique(case.cls[0])) > 1 else float("nan"), "noise"))
        case.share, case.regime = share, what
        _CACHE.clear()          # one case at a time: the large ones hold several N x C fp64 matrices
        _CACHE[name] = (case, _reference(case))
    return _CACHE[name]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the case matrix covers every axis, the comparator rejects simulated faults
# ---------------------------------------------------------------------------------------------------------------------
def test_case_matrix_covers_every_axis():
    vals = lambda i: {v for c in CASES.values() for v in (c[i] if isinstance(c[i], list) else [c[i]])}
    assert {(c + 63) // 64 for c in vals(0)} == {1, 2, 3, 4}
    assert {8, 64, 100, 128, 150, 192, 200, 256} <= vals(0)
    assert {2, 31, 32, 127, 128, 129, 255, 256, 257, 383, 513, 1500, 4000} <= vals(1)
    assert {"one", "two", "ade", "big", "edges"} == vals(2)
    assert {"iid", "straddle", "converged", "hard"} == vals(3)
    assert {0.07, 0.1, 0.5} == vals(4)
    assert {"self", "ms_cs", "ms3", "detach", "eight", "mismatch"} == vals(5)
    assert {0.7, -2.5, 0.0} == vals(6)
    for kb in (3, 4):       # the tile / class edges meet KB = 3 and KB = 4
        assert any((c[0] + 63) // 64 == kb and c[2] == "edges" for c in CASES.values())
        assert any((c[0] + 63) // 64 == kb and c[3] == "straddle" for c in CASES.values())
    assert any(c[5] == "detach" and len(c[1]) == 3 for c in CASES.values())


# cases the fault simulations use (small: the CPU suite evaluates the oracle several times per fault)
FAULT_CASES = ["c150_n383_ade", "c128_n383_ade_ms3", "c100_n255_ade_cs"]


def _got_from_oracle(case, rows_k=None, cls_k=None, self_as_cross=False, neg_pad=0, div_n=None):
    """kernel-like outputs computed by the fp64 oracle under a simulated fault."""
    from oracle import loss_fp64
    terms_out, dF = [], [np.zeros_like(r) for r in case.rows]
    total = 0.0
    for (a, k, self_mask, w, tau, need_dk) in term_list(case.spec, case.S):
        Fk, yk = case.rows[k], case.cls[k]
        if rows_k is not None:          # key columns removed (cross-scale terms: the oracle's self mask needs N1 == N2)
            if not self_mask:
                Fk = rows_k(k, Fk)
                yk = yk[:len(Fk)]
        elif cls_k is not None:
            yk = cls_k(k, yk)
        if neg_pad:
            pad = (-len(Fk)) % 256
            Fk = np.concatenate([Fk, np.zeros((pad, Fk.shape[1]))])
            yk = np.concatenate([yk, np.full(pad, -1)])
        sm = self_mask and not self_as_cross
        loss, dFa, dFk, st = loss_fp64.term(case.rows[a], case.cls[a], Fk, yk, tau, sm, True, 1024)
        P = st["P"]
        div = P if sm else np.where(P > 0, P, 1.0)
        if self_as_cross:
            div = np.where(P > 0, P, 1.0)
        N1 = len(case.rows[a])
        scale_n = 1.0 if div_n is None else N1 / div_n(N1)
        loss *= scale_n
        terms_out.append(dict(neg=st["neg"], possum=st["possum"], S=st["S"], coef_s=st["S"] / (div * N1) * scale_n,
                              coef_pn=st["neg"] / (div * N1) * scale_n, loss=loss))
        total += w * loss
        dF[a] += w * case.g * dFa * scale_n
        if self_mask:
            dF[a] += w * case.g * dFk[:len(case.rows[a])] * scale_n
        elif need_dk:
            m = min(len(dFk), len(case.rows[k]))
            dF[k][:m] += w * case.g * dFk[:m] * scale_n
    return dict(terms=terms_out, total=total, flag=0.0, dF=dF)


def _fault(kind, case, ref):
    if kind == "drop_last_partial_column_tile":
        def cut(k, F):
            n = len(F)
            return F[:n - n % 128] if n % 128 and n > 128 else F
        return _got_from_oracle(case, rows_k=cut)
    if kind == "class_boundary_moved_by_one":
        def move(k, y):
            y = y.copy()
            b = np.nonzero(np.diff(y))[0]
            if len(b):
                j = b[len(b) // 2] + 1          # first row of a class joins the previous class on the key side
                y[j] = y[j - 1]
            return y
        return _got_from_oracle(case, cls_k=move)
    if kind == "diagonal_counted_as_positive":
        return _got_from_oracle(case, self_as_cross=True)
    if kind == "padding_columns_counted_as_negatives":
        return _got_from_oracle(case, neg_pad=1)
    if kind in ("key_side_pass_dropped", "key_side_pass_doubled"):
        got = ref_as_got(ref, case)
        f = 0.0 if kind.endswith("dropped") else 2.0
        from oracle import loss_fp64
        for (a, k, self_mask, w, tau, need_dk) in term_list(case.spec, case.S):
            if need_dk:
                _, _, dFk, _ = loss_fp64.term(case.rows[a], case.cls[a], case.rows[k], case.cls[k], tau, False)
                got["dF"][k] += (f - 1.0) * w * case.g * dFk
        return got
    if kind == "divided_by_upper_bound":
        return _got_from_oracle(case, div_n=lambda n: n + 128)
    if kind == "one_warp_group_scaled":
        got = ref_as_got(ref, case)
        for d in got["dF"]:
            grp = (len(d) - 1) // 32 // 2
            d[32 * grp:32 * grp + 32] *= 1.0 + 2.0 ** -6
        return got
    raise ValueError(kind)


FAULTS = ["drop_last_partial_column_tile", "class_boundary_moved_by_one", "diagonal_counted_as_positive",
          "padding_columns_counted_as_negatives", "key_side_pass_dropped", "key_side_pass_doubled",
          "divided_by_upper_bound", "one_warp_group_scaled"]


@pytest.fixture(scope="module")
def fault_refs():
    return {n: (make_case(n), _reference(make_case(n))) for n in FAULT_CASES}


def test_comparator_accepts_the_bf16_w_emulation(fault_refs):
    """An exact kernel with the bf16 rounding of W passes; so do the fp32 port's statistics (ratio 1 by definition)."""
    for name, (case, ref) in fault_refs.items():
        got = ref_as_got(ref, case)
        fails, worst = compare(ref, got, case.g)
        assert not fails, (name, fails)
        for gt, rt in zip(got["terms"], ref.terms):
            for key in ("neg", "possum", "S"):
                gt[key] = rt["port"][key]
            n1d = rt["div"] * rt["N1"]
            gt["coef_s"], gt["coef_pn"], gt["loss"] = gt["S"] / n1d, gt["neg"] / n1d, rt["port"]["loss"]
        got["total"] = ref.port_total
        fails, worst = compare(ref, got, case.g)
        assert not fails, (name, fails)


@pytest.mark.parametrize("fault", FAULTS)
def test_comparator_rejects_simulated_kernel_faults(fault, fault_refs):
    caught = []
    for name, (case, ref) in fault_refs.items():
        fails, _ = compare(ref, _fault(fault, case, ref), case.g)
        if fails:
            caught.append(f"{name}: {fails[0]}")
    print(f"{fault}: rejected on {len(caught)} of {len(fault_refs)} cases; first: {caught[:1]}")
    assert caught, f"{fault}: no case rejects the simulated fault"


def test_clustered_cases_are_in_the_regime_they_claim():
    """Cheap cases only here (the GPU test asserts the regime of every case before it runs the kernels)."""
    for name, c in CASES.items():
        if c[3] != "iid" and max(c[1]) <= 513:
            case = make_case(name)
            check_regime(case.geom, case.rows[0], case.cls[0], case.tau)


# ---------------------------------------------------------------------------------------------------------------------
# GPU harness
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import mscs_b200
    assert mscs_b200.load().mscs_device_ok() == 1, "libmscs.so needs a compute-capability 10.x device"
    return torch.device("cuda:0")


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _seg(cls, count):
    return np.searchsorted(cls[:count], np.arange(NUM_CLASSES + 1), side="left").astype(np.int32)


def build_device_job(case, dev, upper=None, counts=None, rs=None):
    """mscs_sim_job over synthetic anchor sets.  Without ``upper``: the operand (N_pad, C_pad) bf16, zero-padded to 256
    rows and 64 channels as the gathers write it.  With ``upper`` (per set) and ``counts``: the device-count form --
    rows [count, roundup(count, 256)) zero, rows above NaN (never read), class ids above the count valid but wrong,
    seg from the count, statistics above the count pre-set to a sentinel."""
    from mscs_b200 import _ops
    C_pad = (case.C + 63) // 64 * 64
    sets, samples, keep = [], [], []
    for s in range(case.S):
        n = len(case.rows[s]) if upper is None else upper[s]
        cnt = len(case.rows[s]) if counts is None else counts[s]
        op = torch.zeros(((n + 255) // 256 * 256, C_pad), dtype=torch.bfloat16)
        op[:cnt, :case.C] = torch.from_numpy(case.rows[s][:cnt]).to(torch.bfloat16)
        z_end = (cnt + 255) // 256 * 256
        op[z_end:] = float("nan")
        cls = np.zeros(n, np.int32)
        cls[:cnt] = case.cls[s][:cnt]
        if n > cnt:
            cls[cnt:] = rs.randint(0, NUM_CLASSES, n - cnt)
        op = op.to(dev)
        sets.append(_ops.AnchorSet(N=n, C=case.C, C_pad=C_pad, bf16=op, f32=op[:n].float(),
                                   inv_norm=torch.ones(n, device=dev)))
        samples.append(types.SimpleNamespace(cls=torch.from_numpy(cls).to(dev),
                                             seg=torch.from_numpy(_seg(case.cls[s], cnt)).to(dev)))
    state = _ops.build_job(case.spec, samples, sets, case.terms == "self")
    state.keep += [sets, samples]
    if counts is not None:
        cnt_dev = torch.tensor(counts, dtype=torch.int32, device=dev)
        state.keep.append(cnt_dev)
        stats, coefs = state.keep[0], state.keep[1]
        so = co = 0
        for i, (a, k, *_r) in enumerate(term_list(case.spec, case.S)):
            t = state.job.terms[i]
            t.n1_dev, t.n2_dev = cnt_dev[a].data_ptr(), cnt_dev[k].data_ptr()
            n1 = upper[a]
            for j in range(3):
                stats[so + j * n1 + counts[a]:so + (j + 1) * n1] = 7.0
            for j in range(2):
                coefs[co + j * n1 + counts[a]:co + (j + 1) * n1] = 7.0
            so += 3 * n1
            co += 2 * n1
    return state, sets


def _dF_buffers(sets, dev):
    from mscs_b200 import _lib
    dFs = [torch.zeros((s.N, s.C_pad), dtype=torch.float32, device=dev) for s in sets]
    ptrs = [0] * _lib.MAX_SCALES
    lds = (C.c_int32 * _lib.MAX_SCALES)()
    for i, d in enumerate(dFs):
        ptrs[i], lds[i] = d.data_ptr(), d.shape[1]
    return dFs, _lib.ptr_array(ptrs), lds


def run_forward(state):
    from mscs_b200 import _lib
    _lib.check(_lib.load().mscs_sim_forward(C.byref(state.job), _stream()), "mscs_sim_forward")


def run_backward(state, sets, g, dev, set_mask=None):
    from mscs_b200 import _lib
    lib = _lib.load()
    gt = torch.full((1,), g, dtype=torch.float32, device=dev)
    dFs, ptrs, lds = _dF_buffers(sets, dev)
    if set_mask is None:
        _lib.check(lib.mscs_sim_backward(C.byref(state.job), gt.data_ptr(), ptrs, lds, _stream()), "mscs_sim_backward")
    else:
        for s in range(len(sets)):
            _lib.check(lib.mscs_sim_backward_sets(C.byref(state.job), gt.data_ptr(), ptrs, lds, C.c_uint32(1 << s),
                                                  _stream()), "mscs_sim_backward_sets")
    torch.cuda.synchronize()
    return dFs


def read_outputs(state, case, dFs, counts=None):
    nt = state.job.num_terms
    stats, coefs, out = (t.cpu().double().numpy() for t in state.keep[:3])
    terms, so, co = [], 0, 0
    for i, (a, *_r) in enumerate(term_list(case.spec, case.S)):
        n1 = state.job.terms[i].N1
        c = n1 if counts is None else counts[a]
        terms.append(dict(neg=stats[so:so + c], possum=stats[so + n1:so + n1 + c], S=stats[so + 2 * n1:so + 2 * n1 + c],
                          coef_s=coefs[co:co + c], coef_pn=coefs[co + n1:co + n1 + c], loss=out[i],
                          tail=[stats[so + j * n1 + c:so + (j + 1) * n1] for j in range(3)] +
                               [coefs[co + j * n1 + c:co + (j + 1) * n1] for j in range(2)]))
        so += 3 * n1
        co += 2 * n1
    dF = []
    for s, d in enumerate(dFs):
        c = len(case.rows[s]) if counts is None else counts[s]
        h = d.cpu().double().numpy()
        dF.append(h[:c, :case.C])
        assert np.all(h[:, case.C:] == 0.0), f"set {s}: dF written in the channel padding"
        assert np.all(h[c:] == 0.0), f"set {s}: dF rows at or above the count {c} are not zero"
    return dict(terms=terms, total=out[nt], flag=out[nt + 1], dF=dF)


def _report(case, tag, worst):
    print(f"[{tag}] {case.name}: C={case.C} KB={case.KB} N={case.Ns} layout={case.layout} geometry={case.geom} "
          f"tau={case.tau} terms={case.terms} g={case.g} regime=({case.regime}) share(u>=1/64)={case.share:.3f} "
          f"worst ratio: stats {worst['stats']:.3f} loss {worst['loss']:.3f} dF {worst['dF']:.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_similarity_kernels_vs_fp64_per_row(name, dev):
    case, ref = case_and_ref(name)
    state, sets = build_device_job(case, dev)
    run_forward(state)
    dFs = run_backward(state, sets, case.g, dev)
    got = read_outputs(state, case, dFs)
    fails, worst = compare(ref, got, case.g)
    _report(case, "host counts", worst)
    assert not fails, "\n".join(fails[:12])


DEVCOUNT_CASES = ["c150_n256_edges_ms3", "c150_n129_edges_det", "c256_n257_edges_ms3", "c256_n129_edges",
                  "c100_n256_edges", "c200_n129_mismatch", "c64_n128_two_cs", "c192_n257_one"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", DEVCOUNT_CASES)
def test_device_counts_match_host_counts(name, dev):
    """n1_dev / n2_dev with N1 / N2 as upper bounds far above the counts: rows [count, roundup(count, 256)) zero (as the
    gathers write them), NaN rows above (never read: a read turns up as NaN), valid but wrong class ids above the
    count.  Statistics, losses and dF must match the reference, rows at or above the count keep their initial values
    (statistics) and stay exactly zero (dF)."""
    case, ref = case_and_ref(name)
    rs = np.random.RandomState(5)
    counts = [len(r) for r in case.rows]
    upper = [(c + 255) // 256 * 256 + 256 + 77 for c in counts]
    state, sets = build_device_job(case, dev, upper=upper, counts=counts, rs=rs)
    run_forward(state)
    dFs = run_backward(state, sets, case.g, dev)
    got = read_outputs(state, case, dFs, counts=counts)
    for ti, t in enumerate(got["terms"]):
        for tail in t["tail"]:
            assert np.all(tail == 7.0), f"term {ti}: statistics above the count were written"
    fails, worst = compare(ref, got, case.g)
    _report(case, "device counts", worst)
    assert not fails, "\n".join(fails[:12])


@pytest.mark.gpu
def test_device_count_zero_gives_an_empty_backward(dev):
    """One set with a device count of 0: its dF stays exactly zero, the other set's dF matches the reference of that
    set alone.  (Backward only: an empty forward term has no defined mean.)"""
    case, ref = case_and_ref("c256_n129_edges")
    two = types.SimpleNamespace(**vars(case))
    two.S, two.Ns = 2, case.Ns + [300]
    two.rows = case.rows + [np.full((300, case.C), np.nan)]
    two.cls = case.cls + [np.zeros(300, np.int64)]
    two.spec = make_spec("self", 2, case.tau)
    two.spec.weights = [case.spec.weights[0], 0.5]
    counts, upper = [len(case.rows[0]), 0], [len(case.rows[0]) + 300, 300]
    state, sets = build_device_job(two, dev, upper=upper, counts=counts, rs=np.random.RandomState(3))
    run_forward(state)
    dFs = run_backward(state, sets, case.g, dev)
    assert torch.all(dFs[1] == 0.0), "a set with count 0 received gradient rows"
    d0 = dFs[0].cpu().double().numpy()
    assert np.all(d0[counts[0]:] == 0.0)
    got = read_outputs(state, two, dFs, counts=counts)
    one = dict(terms=got["terms"][:1], total=got["terms"][0]["loss"] * case.spec.weights[0], flag=0.0,
               dF=got["dF"][:1])
    fails, worst = compare(ref, one, case.g)
    _report(case, "count 0 in set 1", worst)
    assert not fails, "\n".join(fails[:12])


RANGE_CASES = ["c150_n1500_big_cs", "c256_n257_edges_ms3", "c128_n383_ade_ms3", "c200_n383_edges_ms3"]


def _pieces(n, bounds):
    edges = [0] + [b for b in bounds if b < n] + [n]
    return [(lo, hi) for lo, hi in zip(edges[:-1], edges[1:])]


@pytest.mark.gpu
@pytest.mark.parametrize("name", RANGE_CASES)
def test_row_ranges_and_set_masks_match_the_full_call(name, dev):
    """What the pooled mode runs: the forward sweeps once per 128-aligned range of anchor rows on the same zeroed
    statistics, then one finalise; the backward once per range of anchor rows and key rows (cross-scale key-side
    pass); and the backward launched once per set bit.  Each must equal the single full call (to fp32 summation order)
    and pass the fp64 comparison.  The ranged backward reads the coefficients of the FULL forward: the ranged forward
    sums its fp32 atomics in another order, a coefficient can move by an ulp, and that flips the bf16 rounding of an
    element of W now and then (one bf16 ulp, up to 2^-7 |W_ij|) -- the inherent bf16-W error the fp64 comparison
    allows, but not "the same call to fp32 summation order"."""
    from mscs_b200 import _lib
    lib = _lib.load()
    case, ref = case_and_ref(name)
    full, sets = build_device_job(case, dev)
    run_forward(full)
    dF_full = run_backward(full, sets, case.g, dev)
    want = read_outputs(full, case, dF_full)

    bounds = [128, 384, 512, 1024]          # uneven 128-aligned pieces
    nt = full.job.num_terms
    st, _ = build_device_job(case, dev)
    terms = term_list(case.spec, case.S)
    npiece = len(bounds) + 1
    for p in range(npiece):
        for i in range(nt):
            t = st.job.terms[i]
            pa = _pieces(t.N1, bounds) + [(t.N1, t.N1)] * npiece
            t.row_begin, t.row_end = pa[p]
            if (t.row_begin, t.row_end) == (0, 0):
                t.row_begin = t.row_end = t.N1
        _lib.check(lib.mscs_sim_forward_sweeps(C.byref(st.job), _stream()), "mscs_sim_forward_sweeps")
    _lib.check(lib.mscs_sim_finalize(C.byref(st.job), _stream()), "mscs_sim_finalize")
    torch.cuda.synchronize()
    fwd = read_outputs(st, case, _dF_buffers(sets, dev)[0])
    st.keep[0].copy_(full.keep[0])          # statistics and coefficients of the full forward (see above)
    st.keep[1].copy_(full.keep[1])
    gt = torch.full((1,), case.g, dtype=torch.float32, device=dev)
    dFs, ptrs, lds = _dF_buffers(sets, dev)
    for p in range(npiece):
        for i in range(nt):
            t = st.job.terms[i]
            pa = _pieces(t.N1, bounds) + [(t.N1, t.N1)] * npiece
            pk = _pieces(t.N2, bounds) + [(t.N2, t.N2)] * npiece
            t.row_begin, t.row_end = pa[p]
            t.krow_begin, t.krow_end = pk[p]
            if (t.row_begin, t.row_end) == (0, 0):
                t.row_begin = t.row_end = t.N1
            if (t.krow_begin, t.krow_end) == (0, 0):
                t.krow_begin = t.krow_end = t.N2
        _lib.check(lib.mscs_sim_backward(C.byref(st.job), gt.data_ptr(), ptrs, lds, _stream()), "mscs_sim_backward")
    torch.cuda.synchronize()
    got = dict(fwd, dF=read_outputs(st, case, dFs)["dF"])
    dF_sets = run_backward(full, sets, case.g, dev, set_mask=True)
    got_sets = read_outputs(full, case, dF_sets)

    for ti, (w_, g_) in enumerate(zip(want["terms"], got["terms"])):
        for key in ("neg", "possum", "S", "coef_s", "coef_pn"):
            np.testing.assert_allclose(g_[key], w_[key], rtol=1e-5, atol=1e-30,
                                       err_msg=f"row ranges, term {ti} {key}")
        assert abs(g_["loss"] - w_["loss"]) <= 1e-5 * abs(w_["loss"])
    for s in range(case.S):
        bound = 64 * EPS32 * ref.absW[s] + 1e-30
        for tag, other in (("row ranges", got), ("set masks", got_sets)):
            e = np.linalg.norm(other["dF"][s] - want["dF"][s], axis=1)
            i = int(np.argmax(e / bound))
            assert np.all(e <= bound), (f"{tag}: set {s} row {i} differs from the full backward by {e[i]:.3e} "
                                        f"(bound {bound[i]:.3e}, |dF| {np.linalg.norm(want['dF'][s][i]):.3e})")
    for tag, other in (("row ranges", got), ("set masks", got_sets)):
        fails, worst = compare(ref, other, case.g)
        _report(case, tag, worst)
        assert not fails, "\n".join(fails[:12])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_end_to_end_clustered_feature_maps(layout, dev):
    """DenseContrastiveLossV2_ms on clustered feature maps (every pixel its class centroid plus noise, not i.i.d.
    noise), C = 150 (KB = 3 end to end), tau = 0.07, against the fp64 oracle on the fp32 maps.  The module rounds the
    unit rows to bf16, the oracle does not, so the comparison adds that rounding to the kernel errors: loss within the
    north-star 1e-3, gradient cosine >= 0.999, the same pixels touched; sampling bit-exact."""
    import mscs_b200
    from mscs_b200 import synth
    from oracle import loss_fp64
    from oracle.config import oracle_cfg
    from oracle.mt19937 import MT19937
    cfg = dict(dataset="CITYSCAPES", experiment=1, temperature=0.07, scales=2, weights=[1.0, 0.6],
               cross_scale_contrast=True, min_views_per_class=5, max_views_per_class=200, max_features_total=3000)
    n, H, W, Cc, strides = 2, 256, 512, 150, [4, 8]
    labels = synth.synth_labels(n, H, W, 19, 6, 16, 0.05, 61)
    rs = np.random.RandomState(62)
    mu = torch.from_numpy(centroids(Cc, "iid", rs)[:20]).float()
    feats = []
    for s in strides:
        lab = labels[:, ::s, ::s]                      # nearest down-sampling at an integer stride (V2.py:194-206)
        # noise 0.13 per channel (norm ~1.6 against the unit centroid): about half of the positive pairs of scale 0
        # have u >= 1/64 at tau = 0.07
        noise = torch.from_numpy(rs.standard_normal((n, Cc) + lab.shape[1:])).float()
        f = mu[lab].permute(0, 3, 1, 2) + 0.13 * noise
        feats.append(f.contiguous())
    torch.manual_seed(7)
    gen = MT19937.from_torch_state(torch.get_rng_state().numpy().tobytes())
    want = loss_fp64.ms_cs_loss(labels.numpy(), [f.double().numpy() for f in feats], oracle_cfg(cfg, 20), gen)
    F0 = want["samples"][0]
    rows0, _ = loss_fp64.gather_normalize(feats[0].double().numpy(), F0["pairs"], F0["idx"])
    y0 = np.repeat(F0["pairs"][:, 1], F0["V"])
    order = np.argsort(y0, kind="stable")
    share, what = check_regime("straddle", rows0[order], y0[order], 0.07)
    mod = mscs_b200.DenseContrastiveLossV2_ms(cfg)
    fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
    fg = [f.to(dev).contiguous(memory_format=fmt).requires_grad_(True) for f in feats]
    torch.manual_seed(7)
    loss = mod(labels.to(dev), fg)
    loss.backward()
    for s, smp in enumerate(mod.last_samples):
        assert np.array_equal(smp.idx_ref.cpu().numpy(), want["samples"][s]["idx"]), "sampled indices differ"
    rel = abs(float(loss) - want["total"]) / abs(want["total"])
    for a, b in zip(list(mod.ms_losses) + list(mod.cs_losses), want["ms"] + want["cs"]):
        assert abs(float(a) - b) <= NORTH_STAR_REL * abs(b)
    line = f"[end to end {layout}] C=150 KB=3 tau=0.07 regime=({what}) share(u>=1/64)={share:.3f} loss rel {rel:.2e}"
    for s, f in enumerate(fg):
        got = f.grad.float().cpu().numpy().astype(np.float64)
        w = want["grads"][s]
        assert np.array_equal(np.abs(got).sum(1) != 0, np.abs(w).sum(1) != 0), "different pixels touched"
        cs_ = cosine(got, w)
        line += f"; scale {s} grad cosine {cs_:.7f}"
        assert cs_ >= 0.999
    print(line)
    assert rel <= NORTH_STAR_REL
