"""CPU reference of the gradients of from_dmxs and from_coords scores (locohd_from_rows_grad, locohd_from_coords_grad).

Row r of A is scored against row r of B.  Each row is sorted stably with its categories, as the oracle does; its first
entry is the anchor and the others are events, walked as one flat scan in (distance, A before B, sorted position)
order with the oracle's weight-function CDF and statistical distance.  With H_k the statistical distance after event
k, dS/dt_k = w(t_k) (H_{k-1} - H_k) (tests/grad_reference.py), so

    G_s[r][c] = g_r w(t) (H_{k-1} - H_k)      for the entry (r, c) of side s that is event k,

and 0 for the anchor's entry, for t = 0 and for non-finite t.  For from_coords, t_ij = |x_j - x_i| enters row i and
row j, so grad_i = sum_j (G[i][j] + G[j][i]) (x_i - x_j) / t_ij.
"""
from __future__ import annotations

import math

import numpy as np

from grad_reference import wf_density


def row_pair_grad(oracle, params, row_a, cat_a, row_b, cat_b, wf_idx=0, g=1.0):
    """(score, grad_a [len(row_a)], grad_b [len(row_b)]) of one row pair, in the rows' own (unsorted) order."""
    C = params.n_categories
    cw = np.ones(C) if params.category_weights is None else np.asarray(params.category_weights, np.float64)
    sd_name, sd_params = params.statistical_distance
    wname, wpar = params.weight_functions[wf_idx]
    rows = [np.asarray(row_a, np.float64), np.asarray(row_b, np.float64)]
    cats = [np.asarray(cat_a, np.int64)[:len(rows[0])], np.asarray(cat_b, np.int64)[:len(rows[1])]]
    order = [np.argsort(r, kind="stable") for r in rows]
    for s in (0, 1):
        if len(rows[s]) == 0:
            raise oracle.OracleError(7)
        if rows[s][order[s][0]] != 0.0:
            raise oracle.OracleError(2)
    counts = [np.zeros(C), np.zeros(C)]
    for s in (0, 1):
        c0 = int(cats[s][order[s][0]])
        if c0 >= C:
            raise oracle.OracleError(3)
        counts[s][c0] += cw[c0]

    def H():
        return oracle.sd_run(sd_name, sd_params, counts[0] / counts[0].sum(), counts[1] / counts[1].sum())

    def W(t):
        return oracle.wf_integral_point(wname, wpar, t)

    grads = [np.zeros(len(rows[0])), np.zeros(len(rows[1]))]
    events = sorted((float(rows[s][order[s][k]]), s, k) for s in (0, 1) for k in range(1, len(rows[s])))
    h = H()
    wprev = W(0.0)
    S = 0.0
    for t, s, k in events:
        w = W(t)
        S += (w - wprev) * h
        wprev = w
        col = int(order[s][k])
        c = int(cats[s][col])
        if c >= C:
            raise oracle.OracleError(3)
        counts[s][c] += cw[c]
        hn = H()
        if g != 0.0 and t > 0.0 and math.isfinite(t):
            grads[s][col] = g * wf_density(wname, wpar, t) * (h - hn)
        h = hn
    S += (W(math.inf) - wprev) * h
    return S, grads[0], grads[1]


def from_rows_grad(oracle, params, rows_a, cat_a, rows_b, cat_b, wf_idx=None, pair_weights=None):
    """(scores [n], grads_a, grads_b): lists of per-row gradient arrays in the rows' own order."""
    scores, ga, gb = [], [], []
    for r in range(len(rows_a)):
        g = 1.0 if pair_weights is None else float(pair_weights[r])
        s, a, b = row_pair_grad(oracle, params, rows_a[r], cat_a, rows_b[r], cat_b,
                                0 if wf_idx is None else int(wf_idx[r]), g)
        scores.append(s)
        ga.append(a)
        gb.append(b)
    return np.array(scores), ga, gb


def euclidean_rows(xyz):
    """t_ij as the device computes it (rows_copy_kernel): sqrt((ex ex + ey ey) + ez ez), 0 on the diagonal."""
    x = np.asarray(xyz, np.float64).reshape(-1, 3)
    e = x[:, None, :] - x[None, :, :]
    return np.sqrt((e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2])


def chain_rule(xyz, G):
    """grad_i = sum_j (G[i][j] + G[j][i]) (x_i - x_j) / t_ij over t_ij > 0."""
    x = np.asarray(xyz, np.float64).reshape(-1, 3)
    t = euclidean_rows(x)
    G = np.asarray(G, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        c = np.where(t > 0, (G + G.T) / np.where(t > 0, t, 1.0), 0.0)
    return (c[:, :, None] * (x[:, None, :] - x[None, :, :])).sum(axis=1)


def from_coords_grad(oracle, params, xyz_a, cat_a, xyz_b, cat_b, wf_idx=None, pair_weights=None):
    """(scores [n], grad_a [n, 3], grad_b [n, 3])."""
    ta, tb = euclidean_rows(xyz_a), euclidean_rows(xyz_b)
    s, ga, gb = from_rows_grad(oracle, params, ta, cat_a, tb, cat_b, wf_idx, pair_weights)
    return s, chain_rule(xyz_a, np.array(ga)), chain_rule(xyz_b, np.array(gb))


# ---- tie-free cases shared by the CPU and GPU tests
def rows_gaps_ok(rows_a, rows_b, kinks=(), gap=1e-3) -> bool:
    """True when, in every row pair, the finite non-anchor entries are at least `gap` apart, from 0 and from every
    kink of the weight function: finite differences of step gap / 100 then see a smooth score."""
    for ra, rb in zip(rows_a, rows_b):
        ra, rb = np.asarray(ra, np.float64), np.asarray(rb, np.float64)
        ev = np.concatenate([np.sort(ra)[1:], np.sort(rb)[1:]])
        ev = np.sort(ev[np.isfinite(ev)])
        if (ev < gap).any() or any((np.abs(ev - k) < gap).any() for k in kinks):
            return False
        if len(ev) > 1 and np.diff(ev).min() < gap:
            return False
    return True


def tie_free_clouds(seed, kinks=(), n=12, C=3, extent=3.2, gap=1e-3):
    """Two clouds of n points (B: A moved by 0.6 A, three categories changed) whose Euclidean rows are tie-free."""
    rng = np.random.default_rng(seed)
    for _ in range(500):
        xa = rng.uniform(-extent, extent, (n, 3))
        xb = xa + rng.normal(0, 0.6, (n, 3))
        ca = rng.integers(0, C, n).astype(np.uint16)
        cb = ca.copy()
        cb[rng.integers(0, n, 3)] = rng.integers(0, C, 3)
        if rows_gaps_ok(euclidean_rows(xa), euclidean_rows(xb), kinks, gap):
            return xa, ca, xb, cb
    raise AssertionError("no tie-free cloud found")


def tie_free_ragged_rows(seed, kinks=(), n_rows=6, C=3, max_len=11, gap=1e-3, hi=8.0):
    """Ragged rows (row r of A and of B of different lengths, 0 at a random place of each) and a category list as
    long as the longest row, tie-free within every row pair."""
    rng = np.random.default_rng(seed)
    for _ in range(500):
        rows = []
        for _side in (0, 1):
            side = []
            for _ in range(n_rows):
                r = rng.uniform(0.2, hi, int(rng.integers(2, max_len + 1)))
                r[rng.integers(0, len(r))] = 0.0
                side.append(r)
            rows.append(side)
        if rows_gaps_ok(rows[0], rows[1], kinks, gap):
            ca = rng.integers(0, C, max_len).astype(np.uint16)
            cb = rng.integers(0, C, max_len).astype(np.uint16)
            return rows[0], ca, rows[1], cb
    raise AssertionError("no tie-free rows found")
