"""locohd_score_within / locohd_score_within_condensed: every pair whose score is at most a bound, as CSR rows on the
device.  The graphs are checked bit for bit against thresholding the dense matrix of locohd_score_cross (between mode)
and the condensed vector of locohd_score_condensed (within mode) on the same ranges and routes; at the bound, with
+inf and NaN scores and with negative and NaN bounds; chunked calls whose storage grows several times against
one-chunk calls (byte for byte); a sample of entries against the CPU oracle (1e-9); scipy's csr_matrix and
connected_components on the result; device copies, repeated calls, the error statuses and the public LoCoHD methods.
"""
import ctypes

import numpy as np
import pytest

from benchdata import synth
from helpers import assert_scores_close, set_both

pytestmark = pytest.mark.gpu

THR = 10.0
ANCH_A = np.arange(0, 320, 23, dtype=np.uint32)   # 14 anchors
ANCH_B = np.arange(3, 320, 17, dtype=np.uint32)   # 19 anchors


def _sets(ctx, clouds, anchors):
    """One structure set of `clouds`; environment e = anchor anchors[e % n] of cloud e // n."""
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    st = ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]), np.concatenate([c.cat for c in clouds]),
                            np.concatenate([c.tag for c in clouds]))
    anchors = np.asarray(anchors, np.uint32)
    env = ctx.envset_build(st, np.tile(anchors, len(clouds)), THR,
                           anchor_struct=np.repeat(np.arange(len(clouds), dtype=np.uint32), len(anchors)))
    return st, env


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint64)


def _take(g):
    """The graph's host CSR arrays; the handle is closed."""
    shape, nnz = g.shape, g.nnz
    ip, ix, sc = g.copy()
    g.close()
    assert ip.shape == (shape[0] + 1,) and ix.shape == sc.shape == (nnz,)
    return ip, ix, sc


def _threshold(M, bound, drop=None):
    """CSR of the entries M[i][j] <= bound (leaving out the `drop` mask): np.nonzero's row-major order."""
    keep = M <= bound
    if drop is not None:
        keep &= ~drop
    r, c = np.nonzero(keep)
    indptr = np.zeros(M.shape[0] + 1, np.uint64)
    indptr[1:] = np.cumsum(keep.sum(axis=1))
    return indptr, c.astype(np.uint32), M[r, c]


def _threshold_condensed(c, n, bound):
    """CSR of the pairs i < j of a condensed vector with c <= bound: row i holds its columns j > i."""
    iu, ju = np.triu_indices(n, 1)
    keep = c <= bound
    indptr = np.zeros(n + 1, np.uint64)
    indptr[1:] = np.cumsum(np.bincount(iu[keep], minlength=n))
    return indptr, ju[keep].astype(np.uint32), c[keep]


def _same(got, want):
    assert np.array_equal(got[0], want[0]), "indptr differs"
    assert np.array_equal(got[1], want[1]), "indices differ"
    assert np.array_equal(_bits(got[2]), _bits(want[2])), "scores differ"


def _self_mask(a_first, n_a, b_first, n_b):
    return (np.arange(n_a)[:, None] + a_first) == (np.arange(n_b)[None, :] + b_first)


@pytest.fixture(scope="module")
def clouds():
    base = synth.gen(31, 40, 8, 7)
    return [synth.partner(base, 1.5, 700 + i) for i in range(3)]


@pytest.mark.parametrize("shape,skip_self", [("inner", False), ("kras_1xn", False), ("nx1", False),
                                             ("same_set", False), ("same_set", True)])
def test_between_equals_the_thresholded_matrix_on_the_tile_route(gpu_ctx, oracle_mod, clouds, shape, skip_self):
    """Ranges that start inside their sets and are no multiple of 4, one row, one column, and A = B with overlapping
    ranges (with and without skip_self): the graph is the thresholded score_cross matrix, scores bit for bit."""
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st_a, env_a = _sets(gpu_ctx, clouds[:2], ANCH_A)
    st_b, env_b = _sets(gpu_ctx, clouds[2:], ANCH_B)
    if shape == "same_set":
        env_b = env_a
    a_first, n_a, b_first, n_b = {"inner": (3, 21, 2, 13), "kras_1xn": (5, 1, 0, len(env_b)),
                                  "nx1": (1, len(env_a) - 1, 7, 1), "same_set": (1, 23, 6, 21)}[shape]
    M, _, _ = gpu_ctx.score_cross(env_a, env_b, a_first, n_a, b_first, n_b)
    drop = _self_mask(a_first, n_a, b_first, n_b) if skip_self else None
    for q in (0.1, 0.5, 1.0):
        bound = float(np.quantile(M, q))
        before = gpu_ctx.tile_launches
        g = gpu_ctx.score_within(env_a, env_b, bound, a_first, n_a, b_first, n_b, skip_self=skip_self)
        assert gpu_ctx.tile_launches > before
        assert g.shape == (n_a, n_b)
        _same(_take(g), _threshold(M, bound, drop))
    for e in (env_a, env_b, st_a, st_b):
        e.close()


PAIR_ROUTE = {
    "no_tiles": dict(n_categories=7),
    "category_weights": dict(n_categories=7, category_weights=np.linspace(0.5, 2.0, 7)),
    "kullback_leibler": dict(n_categories=7, statistical_distance=("Kullback-Leibler", (1e-6,))),
    "c20": dict(n_categories=20),
    "wf_dict": dict(n_categories=7, weight_functions=(("uniform", (3.0, 10.0)), ("kumaraswamy", (2.0, 9.0, 2.0, 3.0)))),
}


@pytest.mark.parametrize("case", sorted(PAIR_ROUTE))
def test_between_equals_the_thresholded_matrix_on_the_pair_route(gpu_ctx, oracle_mod, monkeypatch, case):
    kw = dict(PAIR_ROUTE[case])
    C = kw.pop("n_categories")
    base = synth.gen(41, 40, 8, C)
    members = [synth.partner(base, 1.5, 800 + i) for i in range(2)]
    set_both(gpu_ctx, oracle_mod, C, tag_rule={"accept_same": False}, **kw)
    if case == "no_tiles":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, members, ANCH_A)
    wf = 1 if case == "wf_dict" else 0
    M, _, _ = gpu_ctx.score_cross(env, env, 1, 21, 3, 25, wf_idx=wf)
    for skip_self in (False, True):
        bound = float(np.quantile(M, 0.3))
        before = gpu_ctx.tile_launches
        g = gpu_ctx.score_within(env, env, bound, 1, 21, 3, 25, wf_idx=wf, skip_self=skip_self)
        assert gpu_ctx.tile_launches == before
        _same(_take(g), _threshold(M, bound, _self_mask(1, 21, 3, 25) if skip_self else None))
    env.close(); st.close()


CONDENSED_ROUTE = {
    "tiles": dict(n_categories=7),
    "no_tiles": dict(n_categories=7),
    "kolmogorov_smirnov": dict(n_categories=7, statistical_distance=("Kolmogorov-Smirnov", ())),
    "wf_dict": dict(n_categories=7, weight_functions=(("uniform", (3.0, 10.0)), ("kumaraswamy", (2.0, 9.0, 2.0, 3.0)))),
}


@pytest.mark.parametrize("case", sorted(CONDENSED_ROUTE))
def test_within_equals_the_thresholded_condensed_vector(gpu_ctx, oracle_mod, clouds, monkeypatch, case):
    """Row i carries only its columns j > i, bit for bit the entries of score_condensed on the same range and route;
    n = 0, 1 and 2 give empty graphs of n rows where nothing is scored."""
    kw = dict(CONDENSED_ROUTE[case])
    C = kw.pop("n_categories")
    set_both(gpu_ctx, oracle_mod, C, tag_rule={"accept_same": False}, **kw)
    if case == "no_tiles":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, clouds, ANCH_A)
    wf = 1 if case == "wf_dict" else 0
    for first, n in [(3, 37), (0, 42), (5, 2), (7, 1), (9, 0)]:
        c = gpu_ctx.score_condensed(env, first, n, wf_idx=wf)
        for bound in ([float(np.quantile(c, q)) for q in (0.05, 0.5)] if len(c) else []) + [np.inf]:
            before = gpu_ctx.tile_launches
            g = gpu_ctx.score_within_condensed(env, bound, first, n, wf_idx=wf)
            assert (gpu_ctx.tile_launches > before) == (case == "tiles" and n >= 2)
            assert g.shape == (n, n)
            _same(_take(g), _threshold_condensed(c, n, bound))
    env.close(); st.close()


def test_the_bound_itself_and_negative_and_nan_bounds(gpu_ctx, oracle_mod, clouds):
    from loco_hd_b200._capi import LocoHDError

    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, ANCH_A)
    M, _, _ = gpu_ctx.score_cross(env, env, 2, 30, 0, 40)
    i, j = 7, 11
    ip, ix, sc = _take(gpu_ctx.score_within(env, env, float(M[i, j]), 2, 30, 0, 40))
    assert j in ix[ip[i]:ip[i + 1]]
    _same((ip, ix, sc), _threshold(M, M[i, j]))
    c = gpu_ctx.score_condensed(env, 2, 30)
    got = _take(gpu_ctx.score_within_condensed(env, float(c[100]), 2, 30))
    _same(got, _threshold_condensed(c, 30, c[100]))
    for g in (gpu_ctx.score_within(env, env, -1e-300, 2, 30, 0, 40), gpu_ctx.score_within_condensed(env, -1.0, 2, 30)):
        assert g.nnz == 0
        ip, ix, sc = _take(g)
        assert not ip.any() and len(ix) == len(sc) == 0
    for call in (lambda: gpu_ctx.score_within(env, env, np.nan, 2, 30, 0, 40),
                 lambda: gpu_ctx.score_within_condensed(env, np.nan, 2, 30)):
        with pytest.raises(LocoHDError) as e:
            call()
        assert e.value.status == 10
    env.close(); st.close()


def test_renyi_zero_infinite_and_nan_scores(gpu_ctx, oracle_mod):
    """Renyi alpha = 0 on disjoint compositions gives +inf (the construction of
    test_gpu_grad.py::test_renyi_zero_on_disjoint_compositions: a cloud of category 0 only and the same cloud with
    category 1 only), and NaN where a member lies beyond the weight function's support (a step of zero weight times
    inf): with uniform [0, 9.95] and 10 A environments both occur.  With max_score = inf the +inf entries are in the
    graph and the NaN entries are not."""
    set_both(gpu_ctx, oracle_mod, 2, [("uniform", (0.0, 9.95))], None, ("Renyi", (0.0, 0.0)),
             tag_rule={"accept_same": False})
    base = synth.gen(61, 40, 8, 1)
    zero = synth.partner(base, 0.0, 1)
    zero.cat = np.zeros_like(base.cat)
    one = synth.partner(base, 0.0, 1)
    one.cat = np.ones_like(base.cat)
    st, env = _sets(gpu_ctx, [zero, one, synth.partner(zero, 1.0, 5)], ANCH_A)
    M, _, _ = gpu_ctx.score_cross(env, env)
    assert np.isposinf(M).any() and np.isnan(M).any() and np.isfinite(M).any()
    got = _take(gpu_ctx.score_within(env, env, np.inf))
    _same(got, _threshold(M, np.inf))
    assert np.isposinf(got[2]).any() and not np.isnan(got[2]).any()
    env.close(); st.close()


@pytest.mark.parametrize("route", ["tiles", "pairs"])
def test_chunks_and_growth_change_nothing(gpu_ctx, oracle_mod, clouds, monkeypatch, route):
    """LOCOHD_CROSS_ROWS=4: one chunk per 4 rows.  The bound leaves a whole chunk without an entry (and rows without
    one at chunk edges); with max_score = inf the storage grows several times.  In within mode, 37 rows end with a
    chunk that is only the last row.  Every graph is byte-identical to the one-chunk call."""
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    if route == "pairs":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, clouds, ANCH_A)
    a_first, n_a, n_b = 1, 38, len(env)
    M, _, _ = gpu_ctx.score_cross(env, env, a_first, n_a, 0, n_b)
    own = _self_mask(a_first, n_a, 0, n_b)
    others = np.where(own, np.inf, M)
    block_min = [others[r:r + 4].min() for r in range(0, n_a, 4)]
    bound = float(np.nextafter(max(block_min), -np.inf))   # the chunk with the largest minimum holds no entry
    counts = np.diff(_threshold(M, bound, own)[0].astype(np.int64))
    assert counts.sum() > 0 and any(counts[r:r + 4].sum() == 0 for r in range(0, n_a, 4))
    assert any(counts[r] == 0 and counts[r // 4 * 4:r // 4 * 4 + 4].sum() > 0 for r in range(n_a) if r % 4 in (0, 3))
    for b in (bound, np.inf):
        monkeypatch.delenv("LOCOHD_CROSS_ROWS", raising=False)
        one = _take(gpu_ctx.score_within(env, env, b, a_first, n_a, 0, n_b, skip_self=True))
        monkeypatch.setenv("LOCOHD_CROSS_ROWS", "4")
        launches = gpu_ctx.launch_count
        many = _take(gpu_ctx.score_within(env, env, b, a_first, n_a, 0, n_b, skip_self=True))
        assert gpu_ctx.launch_count - launches >= 10 * 3   # scoring, count and fill for each of the 10 chunks
        _same(many, one)
        _same(one, _threshold(M, b, own))
    for n, chunks in [(38, 10), (37, 9)]:
        monkeypatch.delenv("LOCOHD_CROSS_ROWS", raising=False)
        c = gpu_ctx.score_condensed(env, 1, n)
        for b in (float(np.quantile(c, 0.2)), np.inf):
            monkeypatch.delenv("LOCOHD_CROSS_ROWS", raising=False)
            one = _take(gpu_ctx.score_within_condensed(env, b, 1, n))
            monkeypatch.setenv("LOCOHD_CROSS_ROWS", "4")
            tiles = gpu_ctx.tile_launches
            many = _take(gpu_ctx.score_within_condensed(env, b, 1, n))
            if route == "tiles":
                assert gpu_ctx.tile_launches - tiles == chunks
            _same(many, one)
            _same(one, _threshold_condensed(c, n, b))
    env.close(); st.close()


def test_oracle_scipy_and_connected_components(gpu_ctx, oracle_mod, clouds):
    """A sample of entries against the oracle (1e-9); csr_matrix(...).toarray() is the thresholded matrix where an
    entry is present; connected_components of the upper-triangle graph equals the components of the thresholded
    squareform found by numpy."""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    from scipy.spatial.distance import squareform

    op = set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, ANCH_A)
    n = len(env)
    M, _, _ = gpu_ctx.score_cross(env, env, 0, n, 0, n)
    bound = float(np.quantile(M, 0.25))
    ip, ix, sc = _take(gpu_ctx.score_within(env, env, bound))
    rows = np.repeat(np.arange(n), np.diff(ip.astype(np.int64)))
    sample = np.linspace(0, len(sc) - 1, 40).astype(int)
    want = np.empty(len(sample))
    for k, p in enumerate(sample):
        ca, cb = clouds[rows[p] // len(ANCH_A)], clouds[ix[p] // len(ANCH_A)]
        pair = np.array([[ANCH_A[rows[p] % len(ANCH_A)], ANCH_A[ix[p] % len(ANCH_A)]]], np.uint32)
        want[k] = oracle_mod.from_primitives(op, ca.xyz, ca.cat, ca.tag, cb.xyz, cb.cat, cb.tag, pair, THR)[0]
    assert_scores_close(sc[sample], want)
    D = csr_matrix((sc, ix, ip.astype(np.int64)), shape=(n, n)).toarray()
    keep = M <= bound
    assert np.array_equal(_bits(D[keep]), _bits(M[keep])) and not D[~keep].any()

    c = gpu_ctx.score_condensed(env)
    bound = float(np.quantile(c, 0.02))
    ip, ix, sc = _take(gpu_ctx.score_within_condensed(env, bound))
    G = csr_matrix((sc, ix, ip.astype(np.int64)), shape=(n, n))
    n_comp, labels = connected_components(G, directed=False)
    adj = squareform(c) <= bound
    np.fill_diagonal(adj, False)
    adj |= adj.T
    want = -np.ones(n, np.int64)
    for s in range(n):   # breadth-first search from every unlabelled environment, in index order
        if want[s] >= 0:
            continue
        want[s] = lbl = want.max() + 1
        front = [s]
        while front:
            nxt = np.flatnonzero(adj[front].any(axis=0) & (want < 0))
            want[nxt] = lbl
            front = list(nxt)
    assert n_comp == want.max() + 1 and 1 < n_comp < n
    assert np.array_equal(labels, want)
    assert (G + G.T).nnz == 2 * G.nnz
    env.close(); st.close()


def test_device_copy_determinism_and_errors(gpu_ctx, oracle_mod, clouds, monkeypatch):
    import torch
    from loco_hd_b200._capi import LocoHDError, UNKNOWN_CATEGORY

    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds[:2], ANCH_A)
    st2, other = _sets(gpu_ctx, clouds[2:], ANCH_B)
    n = len(env)
    g = gpu_ctx.score_within(env, env, 0.3, 0, n, 0, n)
    host = g.copy()
    rows, _ = g.shape
    dip = torch.empty(rows + 1, dtype=torch.int64, device="cuda")
    dix = torch.empty(g.nnz, dtype=torch.int32, device="cuda")
    dsc = torch.empty(g.nnz, dtype=torch.float64, device="cuda")
    g.copy(dip.data_ptr(), dix.data_ptr(), dsc.data_ptr())
    _same((dip.cpu().numpy().view(np.uint64), dix.cpu().numpy().view(np.uint32), dsc.cpu().numpy()), host)
    only_scores = g.copy(False, False, None)
    assert only_scores[0] is None and only_scores[1] is None and np.array_equal(_bits(only_scores[2]), _bits(host[2]))
    g.close()
    g.close()   # idempotent
    _same(_take(gpu_ctx.score_within(env, env, 0.3, 0, n, 0, n)), host)
    c1 = _take(gpu_ctx.score_within_condensed(env, 0.3))
    _same(_take(gpu_ctx.score_within_condensed(env, 0.3)), c1)

    lib = gpu_ctx.lib

    def status(fn, *args):
        """Status of a raw call; its output handle must stay NULL."""
        h = ctypes.c_void_p(1)
        st_ = fn(gpu_ctx.h, *args, ctypes.byref(h))
        assert st_ and h.value is None
        return st_

    w = lib.locohd_score_within
    wc = lib.locohd_score_within_condensed
    assert status(w, env.h, n - 3, 4, env.h, 0, 8, 0, 0, 1.0) == 8
    assert status(w, env.h, 0, 4, env.h, n + 1, 0, 0, 0, 1.0) == 8
    assert status(w, env.h, 0, 4, env.h, 0, n + 1, 0, 0, 1.0) == 8
    assert status(w, env.h, 0, 4, other.h, 0, 8, 0, 1, 1.0) == 10     # skip_self with two sets
    assert status(w, env.h, 0, 4, env.h, 0, 8, 1, 0, 1.0) == 10       # weight function index
    assert status(w, env.h, 0, 4, env.h, 0, 8, 0, 0, float("nan")) == 10
    assert status(wc, env.h, n - 3, 4, 0, 1.0) == 8
    assert status(wc, env.h, 0, n + 1, 0, 1.0) == 8
    assert status(wc, env.h, 0, 8, 1, 1.0) == 10
    for sd in [("Kullback-Leibler", (1e-6,)), ("Renyi", (1.7, 0.2))]:
        set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False}, statistical_distance=sd)
        st4, env4 = _sets(gpu_ctx, clouds[:1], ANCH_A)
        with pytest.raises(LocoHDError, match="symmetric") as e:
            gpu_ctx.score_within_condensed(env4, 1.0, 0, 8)
        assert e.value.status == 10
        _take(gpu_ctx.score_within(env4, env4, 1.0, 0, 8, 0, 8))   # both triangles are fine
        env4.close(); st4.close()
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    bad = synth.partner(clouds[0], 0.5, 77)
    bad.cat = bad.cat.copy()
    bad.cat[ANCH_A[2] + 1] = UNKNOWN_CATEGORY
    st3, env3 = _sets(gpu_ctx, [clouds[1], bad], ANCH_A)
    for no_tiles in ("0", "1"):
        monkeypatch.setenv("LOCOHD_NO_TILES", no_tiles)
        assert status(w, env3.h, 0, len(env3), env3.h, 0, 8, 0, 0, 1.0) == 3
        assert status(wc, env3.h, 0, len(env3), 0, 1.0) == 3
    gpu_ctx.synchronize()   # the context is usable afterwards
    for e in (env, other, env3, st, st2, st3):
        e.close()


def test_public_methods_equal_the_c_abi(gpu_ctx, oracle_mod, clouds):
    """LoCoHD.environments_within / environments_within_condensed equal the C-ABI graphs as int64 / uint32 / float64
    host arrays; bad ranges, weight functions, exclude_self with two sets, a NaN bound and an asymmetric distance in
    within mode raise ValueError."""
    import loco_hd

    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, ANCH_A)
    cats = [f"T{i}" for i in range(7)]
    lchd = loco_hd.LoCoHD(cats, loco_hd.WeightFunction("uniform", [3.0, 10.0]),
                          loco_hd.TagPairingRule({"accept_same": False}))
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    xyz, cat, tag = (np.concatenate([getattr(c, f) for c in clouds]) for f in ("xyz", "cat", "tag"))
    pst = lchd.structures(offs, xyz, cat, tag)
    penv = lchd.environments(pst, np.tile(ANCH_A, len(clouds)), THR,
                             anchor_struct=np.repeat(np.arange(len(clouds), dtype=np.uint32), len(ANCH_A)))
    ip, ix, sc = lchd.environments_within(penv, penv, 0.3, a_range=(3, 30), b_range=(1, 40), exclude_self=True)
    assert ip.dtype == np.int64 and ix.dtype == np.uint32 and sc.dtype == np.float64
    _same((ip.view(np.uint64), ix, sc), _take(gpu_ctx.score_within(env, env, 0.3, 3, 27, 1, 39, skip_self=True)))
    ip, ix, sc = lchd.environments_within_condensed(penv, 0.3, env_range=(2, 35))
    _same((ip.view(np.uint64), ix, sc), _take(gpu_ctx.score_within_condensed(env, 0.3, 2, 33)))
    ip, ix, sc = lchd.environments_within_condensed(penv, 0.3, env_range=(4, 5))
    assert np.array_equal(ip, [0, 0]) and len(ix) == len(sc) == 0
    for bad in [dict(a_range=(-1, 3)), dict(a_range=(5, 4)), dict(b_range=(0, len(env) + 1)), dict(wf_idx=1),
                dict(wf_idx=-1), dict(max_score=float("nan"))]:
        kw = dict(max_score=0.3)
        kw.update(bad)
        with pytest.raises(ValueError):
            lchd.environments_within(penv, penv, **kw)
    for bad in [dict(env_range=(-1, 3)), dict(env_range=(0, len(env) + 1)), dict(wf_idx=1),
                dict(max_score=float("nan"))]:
        kw = dict(max_score=0.3)
        kw.update(bad)
        with pytest.raises(ValueError):
            lchd.environments_within_condensed(penv, **kw)
    other = lchd.environments(pst, ANCH_A, THR)
    with pytest.raises(ValueError):
        lchd.environments_within(penv, other, 0.3, exclude_self=True)
    kl = loco_hd.LoCoHD(cats, loco_hd.WeightFunction("uniform", [3.0, 10.0]),
                        loco_hd.TagPairingRule({"accept_same": False}),
                        statistical_distance=loco_hd.StatisticalDistance("Kullback-Leibler", [1e-6]))
    kst = kl.structures(offs, xyz, cat, tag)
    kenv = kl.environments(kst, ANCH_A, THR)
    with pytest.raises(ValueError, match="symmetric"):
        kl.environments_within_condensed(kenv, 0.3)
    assert len(kl.environments_within(kenv, kenv, np.inf)[1]) == len(ANCH_A) ** 2
    for e in (penv, other, pst, kenv, kst, env, st):
        e.close()
