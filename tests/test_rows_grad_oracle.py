"""CPU checks of the reference (tests/rows_grad_reference.py) that the GPU's locohd_from_rows_grad and
locohd_from_coords_grad are compared with: per-entry gradients against central finite differences of oracle.from_dmxs
(and, for ragged rows, of oracle.from_anchors on the co-sorted rows), coordinate gradients against central finite
differences of oracle.from_coords."""
import numpy as np
import pytest

import rows_grad_reference as rr
from grad_reference import H, SDS, WFS, kinks

N = 9   # points / rows per case


def params(oracle_mod, wfs, sd, cat_w):
    return oracle_mod.Params(3, [(n, list(p)) for n, p in wfs], cat_w, (sd[0], list(sd[1])), None)


def case_kind(wf, sd):
    k = sorted(WFS).index(wf) + 4 * sorted(SDS).index(sd)
    cat_w = None if k % 2 == 0 else [0.6, 1.7, 1.1]
    weights = np.linspace(-0.7, 1.9, N) if k % 4 == 1 else None
    if weights is not None:
        weights[3] = 0.0
    return k, cat_w, weights


def close_to_fd(got, fd):
    scale = max(float(np.abs(np.concatenate([np.ravel(f) for f in fd])).max()), 1e-300)
    err = max(float(np.abs(np.ravel(g) - np.ravel(f)).max()) for g, f in zip(got, fd))
    assert scale > 0 and err <= 1e-6 * scale, f"gradient vs finite differences: {err} (max |g| {scale})"


def dmx_finite_differences(oracle_mod, op, ta, ca, tb, cb, wf_idx, weights):
    w = np.ones(len(ta)) if weights is None else weights

    def f(a, b):
        return float(np.dot(w, oracle_mod.from_dmxs(op, ca, cb, a, b, wf_idx=wf_idx)))
    out = []
    for side in (0, 1):
        g = np.zeros_like(ta)
        for r in range(g.shape[0]):
            for c in range(g.shape[1]):
                if r == c:
                    continue   # the anchor entry: its 0 is required
                m = [ta.copy(), tb.copy()]
                m[side][r, c] += H
                fp = f(*m)
                m[side][r, c] -= 2 * H
                g[r, c] = (fp - f(*m)) / (2 * H)
        out.append(g)
    return out


@pytest.mark.parametrize("wf", sorted(WFS))
@pytest.mark.parametrize("sd", sorted(SDS))
def test_entry_gradients_match_finite_differences_of_from_dmxs(oracle_mod, wf, sd):
    """Every weight-function family x every statistical distance; category weights and pair weights (with a 0 and
    negative values) vary with the case.  Rows: Euclidean matrices of tie-free clouds, perturbed entry by entry."""
    k, cat_w, weights = case_kind(wf, sd)
    op = params(oracle_mod, [WFS[wf]], SDS[sd], cat_w)
    xa, ca, xb, cb = rr.tie_free_clouds(200 + k, kinks([WFS[wf]]), n=N)
    ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
    s, ga, gb = rr.from_rows_grad(oracle_mod, op, ta, ca, tb, cb, pair_weights=weights)
    assert np.abs(s - oracle_mod.from_dmxs(op, ca, cb, ta, tb)).max() <= 1e-12
    ga, gb = np.array(ga), np.array(gb)
    assert not np.diagonal(ga).any() and not np.diagonal(gb).any()
    close_to_fd((ga, gb), dmx_finite_differences(oracle_mod, op, ta, ca, tb, cb, None, weights))


@pytest.mark.parametrize("wf", sorted(WFS))
@pytest.mark.parametrize("sd", sorted(SDS))
def test_coordinate_gradients_match_finite_differences_of_from_coords(oracle_mod, wf, sd):
    k, cat_w, weights = case_kind(wf, sd)
    op = params(oracle_mod, [WFS[wf]], SDS[sd], cat_w)
    xa, ca, xb, cb = rr.tie_free_clouds(300 + k, kinks([WFS[wf]]), n=N)
    s, ga, gb = rr.from_coords_grad(oracle_mod, op, xa, ca, xb, cb, pair_weights=weights)
    assert np.abs(s - oracle_mod.from_coords(op, ca, cb, xa, xb)).max() <= 1e-12
    w = np.ones(N) if weights is None else weights
    fd = []
    for side in (0, 1):
        g = np.zeros((N, 3))
        for i in range(N):
            for q in range(3):
                x = [xa.copy(), xb.copy()]
                x[side][i, q] += H
                fp = float(np.dot(w, oracle_mod.from_coords(op, ca, cb, *x)))
                x[side][i, q] -= 2 * H
                g[i, q] = (fp - float(np.dot(w, oracle_mod.from_coords(op, ca, cb, *x)))) / (2 * H)
        fd.append(g)
    close_to_fd((ga, gb), fd)


@pytest.mark.parametrize("sd", ["Hellinger", "Kullback-Leibler"])
def test_per_row_weight_functions(oracle_mod, sd):
    wfs = [WFS[w] for w in sorted(WFS)]
    op = params(oracle_mod, wfs, SDS[sd], [1.3, 0.4, 0.9])
    xa, ca, xb, cb = rr.tie_free_clouds(7, kinks(wfs), n=N)
    ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
    wf_idx = (np.arange(N) % 4).astype(np.int32)
    weights = np.linspace(-0.7, 1.9, N)
    s, ga, gb = rr.from_rows_grad(oracle_mod, op, ta, ca, tb, cb, wf_idx=wf_idx, pair_weights=weights)
    assert np.abs(s - oracle_mod.from_dmxs(op, ca, cb, ta, tb, wf_idx=wf_idx)).max() <= 1e-12
    close_to_fd((np.array(ga), np.array(gb)),
                dmx_finite_differences(oracle_mod, op, ta, ca, tb, cb, wf_idx, weights))


@pytest.mark.parametrize("sd", ["Hellinger", "Renyi"])
def test_ragged_rows_match_finite_differences_of_from_anchors(oracle_mod, sd):
    """Rows of different lengths, each co-sorted with the first len(row) categories (as from_dmxs does)."""
    op = params(oracle_mod, [WFS["kumaraswamy"]], SDS[sd], [0.6, 1.7, 1.1])
    ra, ca, rb, cb = rr.tie_free_ragged_rows(17, kinks([WFS["kumaraswamy"]]))
    weights = np.linspace(-0.7, 1.9, len(ra))

    def score(a, b):
        oa, ob = np.argsort(a, kind="stable"), np.argsort(b, kind="stable")
        return oracle_mod.from_anchors(op, ca[:len(a)][oa], cb[:len(b)][ob], a[oa], b[ob])
    s, ga, gb = rr.from_rows_grad(oracle_mod, op, ra, ca, rb, cb, pair_weights=weights)
    fd_a, fd_b = [], []
    for r in range(len(ra)):
        assert abs(s[r] - score(ra[r], rb[r])) <= 1e-12
        for row, other, out, first in ((ra[r], rb[r], fd_a, True), (rb[r], ra[r], fd_b, False)):
            g = np.zeros(len(row))
            for c in np.flatnonzero(row != 0.0):
                x = row.copy()
                x[c] += H
                fp = score(x, other) if first else score(other, x)
                x[c] -= 2 * H
                fm = score(x, other) if first else score(other, x)
                g[c] = weights[r] * (fp - fm) / (2 * H)
            out.append(g)
    close_to_fd((np.concatenate(ga), np.concatenate(gb)), (np.concatenate(fd_a), np.concatenate(fd_b)))
    for r in range(len(ra)):   # the anchor entries
        assert ga[r][np.argmin(ra[r])] == 0.0 and gb[r][np.argmin(rb[r])] == 0.0


@pytest.mark.parametrize("sd", ["Hellinger", "Kullback-Leibler"])
def test_infinite_entries_give_exact_zeros(oracle_mod, sd):
    """Banned entries (+inf, as compare_ensembles.py writes them) get exactly 0 and leave the finite entries'
    gradients as those of the rows without them."""
    op = params(oracle_mod, [("uniform", [3.0, 10.0])], SDS[sd], None)
    xa, ca, xb, cb = rr.tie_free_clouds(23, kinks([("uniform", [3.0, 10.0])]), n=N)
    ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
    ban = np.random.default_rng(1).random(ta.shape) < 0.3
    np.fill_diagonal(ban, False)
    ia, ib = np.where(ban, np.inf, ta), np.where(ban.T, np.inf, tb)
    s, ga, gb = rr.from_rows_grad(oracle_mod, op, ia, ca, ib, cb)
    assert np.isfinite(s).all()
    assert np.abs(s - oracle_mod.from_dmxs(op, ca, cb, ia, ib)).max() <= 1e-12
    ga, gb = np.array(ga), np.array(gb)
    assert (ga[ban] == 0.0).all() and (gb[ban.T] == 0.0).all()
    assert np.isfinite(ga).all() and np.isfinite(gb).all()
    close_to_fd((ga, gb), dmx_finite_differences(oracle_mod, op, ia, ca, ib, cb, None, None))
