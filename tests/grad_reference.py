"""CPU reference of the coordinate gradients of LoCoHD scores (locohd_from_primitives_grad).

It uses the oracle's own environments (``oracle.environment``), its weight-function CDF and statistical distances, and
walks the non-anchor members of both environments as one flat scan in (distance, A before B, environment order)
order.  With H_k the statistical distance after event k,

    S = sum_k (W(t_k) - W(t_{k-1})) H_{k-1} + (W(inf) - W(t_K)) H_K,     dS/dt_k = w(t_k) (H_{k-1} - H_k),

and dt/dx_member = (x_member - x_anchor) / t = -dt/dx_anchor.  The density w = W' is written out here for the four
weight-function families (``wf_density``); tests check it against numerical derivatives of the oracle's CDF and
check the gradients against finite differences of the oracle's scores.
"""
from __future__ import annotations

import math

import numpy as np


def wf_density(name: str, params, x: float) -> float:
    """w(x) = dW/dx with the comparisons of the CDF at the kinks (x < x_min -> 0, x > x_max -> 0)."""
    p = [float(v) for v in params]
    if name == "hyper_exp":
        half = len(p) // 2
        a, b = p[:half], p[half:2 * half]
        return sum(ai * bi * math.exp(-bi * x) for ai, bi in zip(a, b)) / sum(a)
    if name == "dagum":
        a, b, q = p[0], p[1], p[2]
        if x <= 0.0:
            return 0.0 if a * q > 1.0 else (a * q / b if a * q == 1.0 else math.inf)
        lu = -a * (math.log(x) - math.log(b))   # log u, u = (x / b)^-a, W = (1 + u)^-q
        l = -q * lu - (q + 1.0) * math.log1p(math.exp(-lu)) if lu > 0 else lu - (q + 1.0) * math.log1p(math.exp(lu))
        return math.exp(l + math.log(a * q) - math.log(x))   # a q / x inside: no inf * 0 for tiny x
    lo, hi = p[0], p[1]
    if x < lo or x > hi:
        return 0.0
    if name == "uniform":
        return 1.0 / (hi - lo)
    if name == "kumaraswamy":
        a, b = p[2], p[3]
        z = (x - lo) / (hi - lo)
        return a * b * z ** (a - 1.0) * (1.0 - z ** a) ** (b - 1.0) / (hi - lo)
    raise ValueError(name)


def from_primitives_grad(oracle, params, xyz_a, cat_a, tag_a, xyz_b, cat_b, tag_b, anchors, threshold: float,
                         wf_idx=None, pair_weights=None):
    """(scores [P], grad_a [n_a, 3], grad_b [n_b, 3]) with grad = sum_p pair_weights[p] dS_p / dxyz."""
    xyz = [np.asarray(xyz_a, np.float64).reshape(-1, 3), np.asarray(xyz_b, np.float64).reshape(-1, 3)]
    cats = [np.asarray(cat_a, np.uint16), np.asarray(cat_b, np.uint16)]
    tags = [np.asarray(tag_a, np.uint32), np.asarray(tag_b, np.uint32)]
    anchors = np.asarray(anchors, np.int64).reshape(-1, 2)
    P = len(anchors)
    C = params.n_categories
    cw = np.ones(C) if params.category_weights is None else np.asarray(params.category_weights, np.float64)
    sd_name, sd_params = params.statistical_distance
    scores = np.zeros(P)
    grad = [np.zeros_like(xyz[0]), np.zeros_like(xyz[1])]
    for p in range(P):
        wname, wpar = params.weight_functions[0 if wf_idx is None else int(wf_idx[p])]
        W = lambda t: oracle.wf_integral_point(wname, wpar, t)   # noqa: E731
        g = 1.0 if pair_weights is None else float(pair_weights[p])
        envs = [oracle.environment(params, xyz[s], cats[s], tags[s], int(anchors[p, s]), threshold) for s in (0, 1)]
        if len(envs[0][0]) == 0 or len(envs[1][0]) == 0:
            raise oracle.OracleError(7)
        counts = [np.zeros(C), np.zeros(C)]
        for s in (0, 1):
            c0 = int(envs[s][2][0])
            if c0 >= C:
                raise oracle.OracleError(3)
            counts[s][c0] += cw[c0]

        def H():
            return oracle.sd_run(sd_name, sd_params, counts[0] / counts[0].sum(), counts[1] / counts[1].sum())

        events = sorted((float(envs[s][1][k]), s, k) for s in (0, 1) for k in range(1, len(envs[s][0])))
        h = H()
        wprev = W(max(float(envs[0][1][0]), float(envs[1][1][0])))
        S = 0.0
        for t, s, k in events:
            w = W(t)
            S += (w - wprev) * h
            wprev = w
            c = int(envs[s][2][k])
            if c >= C:
                raise oracle.OracleError(3)
            counts[s][c] += cw[c]
            hn = H()
            if g != 0.0 and t > 0.0:
                m, a = int(envs[s][0][k]), int(anchors[p, s])
                v = g * wf_density(wname, wpar, t) * (h - hn) / t * (xyz[s][m] - xyz[s][a])
                grad[s][m] += v
                grad[s][a] -= v
            h = hn
        S += (W(math.inf) - wprev) * h
        scores[p] = S
    return scores, grad[0], grad[1]


def event_gaps_ok(xyz_a, xyz_b, anchors, threshold: float, kinks=(), gap: float = 1e-3) -> bool:
    """True when finite differences of step h = gap / 100 see a smooth score: no two merged events of a pair, no
    member and its anchor, and no distance and the threshold or a kink of the weight function lie within `gap`."""
    xyz = [np.asarray(xyz_a, np.float64).reshape(-1, 3), np.asarray(xyz_b, np.float64).reshape(-1, 3)]
    anchors = np.asarray(anchors, np.int64).reshape(-1, 2)
    for p in range(len(anchors)):
        ev = []
        for s in (0, 1):
            d = np.sqrt(((xyz[s] - xyz[s][anchors[p, s]]) ** 2).sum(axis=1))
            d = np.delete(d, anchors[p, s])
            if (np.abs(d - threshold) < gap).any() or (d < gap).any():
                return False
            for k in kinks:
                if (np.abs(d - k) < gap).any():
                    return False
            ev.append(d[d < threshold])
        merged = np.sort(np.concatenate(ev))
        if len(merged) > 1 and np.diff(merged).min() < gap:
            return False
    return True


# ---- cases shared by the CPU and GPU gradient tests
WFS = {
    "hyper_exp": ("hyper_exp", [1.0, 2.0, 0.5, 0.15]),
    "dagum": ("dagum", [2.5, 3.0, 1.3]),
    "uniform": ("uniform", [1.5, 5.0]),
    "kumaraswamy": ("kumaraswamy", [1.0, 5.5, 2.3, 1.7]),
}
SDS = {
    "Hellinger": ("Hellinger", [2.0]),
    "Hellinger-e": ("Hellinger", [3.26]),
    "Kolmogorov-Smirnov": ("Kolmogorov-Smirnov", []),
    "Kullback-Leibler": ("Kullback-Leibler", [0.3]),
    "Renyi": ("Renyi", [1.7, 0.2]),
}
THRESHOLD = 6.0
H = 1e-5


def kinks(wfs):
    return [v for name, p in wfs if name in ("uniform", "kumaraswamy") for v in p[:2]]


def tie_free_case(seed, wfs, n=14, C=3, n_tags=3, extent=3.2, gap=100 * H):
    """A random pair of small clouds (B: A moved by 0.6 A and three categories changed, anchors every third
    primitive) whose events are at least `gap` apart, regenerated until they are."""
    rng = np.random.default_rng(seed)
    for _ in range(200):
        A = (rng.uniform(-extent, extent, (n, 3)), rng.integers(0, C, n).astype(np.uint16),
             rng.integers(0, n_tags, n).astype(np.uint32))
        B = (A[0] + rng.normal(0, 0.6, (n, 3)), A[1].copy(), A[2].copy())
        B[1][rng.integers(0, n, 3)] = rng.integers(0, C, 3)
        anchors = np.stack([np.arange(0, n, 3), np.arange(0, n, 3)], axis=1).astype(np.uint32)
        if event_gaps_ok(A[0], B[0], anchors, THRESHOLD, kinks(wfs), gap=gap):
            return A, B, anchors
    raise AssertionError("no tie-free cloud found")
