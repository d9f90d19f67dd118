"""locohd_score_cross: every environment of a range of one env-set against every environment of a range of another -
the score matrix and its k nearest columns per row.  The matrix is checked against the CPU oracle on the anchor pairs
it stands for (1e-9), against locohd_score_pairs on the explicit pair list (the tile kernel within 1e-12, the pair
kernel bit for bit), the k nearest against a stable numpy sort of the matrix the same call returns, chunked calls
against one-chunk calls (bit for bit), and the error statuses and the public LoCoHD methods.
"""
import numpy as np
import pytest

from benchdata import synth
from helpers import assert_scores_close, set_both

pytestmark = pytest.mark.gpu

THR = 10.0


def _sets(ctx, clouds, anchors):
    """One structure set of `clouds`; environment e = anchor anchors[e % n] of cloud e // n."""
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    st = ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]), np.concatenate([c.cat for c in clouds]),
                            np.concatenate([c.tag for c in clouds]))
    anchors = np.asarray(anchors, np.uint32)
    env = ctx.envset_build(st, np.tile(anchors, len(clouds)), THR,
                           anchor_struct=np.repeat(np.arange(len(clouds), dtype=np.uint32), len(anchors)))
    return st, env


def _oracle_matrix(oracle, op, clouds_a, anch_a, rows, clouds_b, anch_b, cols):
    """Oracle scores of environment rows[i] (of the set built from clouds_a / anch_a) against cols[j]."""
    M = np.empty((len(rows), len(cols)))
    for i, ea in enumerate(rows):
        ca, pa = clouds_a[ea // len(anch_a)], anch_a[ea % len(anch_a)]
        for cb in range(len(clouds_b)):
            js = [j for j, eb in enumerate(cols) if eb // len(anch_b) == cb]
            if not js:
                continue
            pairs = np.array([(pa, anch_b[cols[j] % len(anch_b)]) for j in js], np.uint32)
            b = clouds_b[cb]
            M[i, js] = oracle.from_primitives(op, ca.xyz, ca.cat, ca.tag, b.xyz, b.cat, b.tag, pairs, THR)
    return M


def _pair_list(a_first, n_a, b_first, n_b):
    i, j = np.meshgrid(np.arange(n_a) + a_first, np.arange(n_b) + b_first, indexing="ij")
    return np.stack([i.ravel(), j.ravel()], axis=1).astype(np.uint32)


@pytest.fixture(scope="module")
def clouds():
    base = synth.gen(31, 40, 8, 7)
    members = [synth.partner(base, 1.5, 700 + i) for i in range(3)]
    return base, members


ANCH_A = np.arange(0, 320, 23, dtype=np.uint32)   # 14 anchors
ANCH_B = np.arange(3, 320, 17, dtype=np.uint32)   # 19 anchors


@pytest.mark.parametrize("shape", ["inner", "kras_1xn", "nx1", "same_set"])
def test_matrix_equals_the_oracle(gpu_ctx, oracle_mod, clouds, shape):
    """Ranges that start inside their sets and are no multiple of 4, the one-anchor-against-all shape of
    kras_scan.py:47-52, one column, and A = B: every entry against the oracle's score of its anchor pair."""
    _, members = clouds
    op = set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    ca, cb = members[:2], members[2:]
    st_a, env_a = _sets(gpu_ctx, ca, ANCH_A)
    st_b, env_b = _sets(gpu_ctx, cb, ANCH_B)
    if shape == "same_set":
        env_b, cb, anch_b = env_a, ca, ANCH_A
    else:
        anch_b = ANCH_B
    a_first, n_a, b_first, n_b = {"inner": (3, 21, 2, 13), "kras_1xn": (5, 1, 0, len(env_b)),
                                  "nx1": (0, len(env_a), 7, 1), "same_set": (1, 23, 0, len(env_a))}[shape]
    M, _, _ = gpu_ctx.score_cross(env_a, env_b, a_first, n_a, b_first, n_b)
    assert M.shape == (n_a, n_b)
    want = _oracle_matrix(oracle_mod, op, ca, ANCH_A, list(range(a_first, a_first + n_a)), cb, anch_b,
                          list(range(b_first, b_first + n_b)))
    assert_scores_close(M.ravel(), want.ravel())
    for e in (env_a, env_b, st_a, st_b):
        e.close()


def test_tile_route_equals_score_pairs(gpu_ctx, oracle_mod, clouds):
    """W-keyed sets, Hellinger-2, unit weights: the tile kernel (counted by tile_launches) within 1e-12 of the pair
    kernel on the explicit pair list - the tolerance between the two kernels on job lists."""
    _, members = clouds
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, members, ANCH_A)
    before = gpu_ctx.tile_launches
    M, _, _ = gpu_ctx.score_cross(env, env, 2, 37, 5, 30)
    assert gpu_ctx.tile_launches > before
    before = gpu_ctx.tile_launches
    ref = gpu_ctx.score_pairs(env, env, _pair_list(2, 37, 5, 30))
    assert gpu_ctx.tile_launches == before
    assert np.abs(M.ravel() - ref).max() <= 1e-12
    env.close(); st.close()


PAIR_ROUTE = {
    "no_tiles": dict(n_categories=7),
    "category_weights": dict(n_categories=7, category_weights=np.linspace(0.5, 2.0, 7)),
    "kullback_leibler": dict(n_categories=7, statistical_distance=("Kullback-Leibler", (1e-6,))),
    "c20": dict(n_categories=20),
    "wf_dict": dict(n_categories=7, weight_functions=(("uniform", (3.0, 10.0)), ("kumaraswamy", (2.0, 9.0, 2.0, 3.0)))),
}


@pytest.mark.parametrize("case", sorted(PAIR_ROUTE))
def test_pair_route_equals_score_pairs_bit_for_bit(gpu_ctx, oracle_mod, monkeypatch, case):
    """Configurations the tile kernel does not take (and LOCOHD_NO_TILES): explicit pairs on the pair kernel, the
    same kernel and arithmetic as score_pairs, so the matrix is bit-identical to it."""
    kw = dict(PAIR_ROUTE[case])
    C = kw.pop("n_categories")
    base = synth.gen(41, 40, 8, C)
    members = [synth.partner(base, 1.5, 800 + i) for i in range(2)]
    set_both(gpu_ctx, oracle_mod, C, tag_rule={"accept_same": False}, **kw)
    if case == "no_tiles":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, members, ANCH_A)
    wf = 1 if case == "wf_dict" else 0
    before = gpu_ctx.tile_launches
    M, _, _ = gpu_ctx.score_cross(env, env, 1, 21, 3, 25, wf_idx=wf)
    assert gpu_ctx.tile_launches == before
    pairs = _pair_list(1, 21, 3, 25)
    ref = gpu_ctx.score_pairs(env, env, pairs, wf_idx=np.full(len(pairs), wf, np.uint32))
    assert np.array_equal(M.ravel().view(np.uint64), ref.view(np.uint64))
    env.close(); st.close()


def _knn_reference(M, k, a_first, b_first, skip_self):
    idx = np.empty((M.shape[0], k), np.int64)
    for i in range(M.shape[0]):
        cols = np.arange(M.shape[1])
        if skip_self:
            cols = cols[cols + b_first != a_first + i]
        idx[i] = cols[np.argsort(M[i, cols], kind="stable")[:k]]
    return idx


@pytest.mark.parametrize("route", ["tiles", "pairs"])
@pytest.mark.parametrize("k,skip_self", [(1, False), (5, True), (32, False), (32, True)])
def test_nearest_equal_a_stable_sort_of_the_matrix(gpu_ctx, oracle_mod, clouds, monkeypatch, route, k, skip_self):
    """Duplicated structures give exactly equal scores (ties ordered by column); skip_self leaves out each row's own
    environment; the k-nearest-only call (matrix kept on the device) gives the same lists."""
    base, members = clouds
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    if route == "pairs":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, [members[0], members[1], members[0]], ANCH_A)   # 42 environments, 14 duplicated
    a_first, n_a, b_first, n_b = 4, 30, 2, 40
    M, ks, ki = gpu_ctx.score_cross(env, env, a_first, n_a, b_first, n_b, skip_self=skip_self, k=k)
    want = _knn_reference(M, k, a_first, b_first, skip_self)
    assert np.array_equal(ki.astype(np.int64), want)
    assert np.array_equal(ks.view(np.uint64), np.take_along_axis(M, want, axis=1).view(np.uint64))
    if k > 1:
        assert (ks[:, 0] == ks[:, 1]).any(), "the duplicated structures must produce ties"
    _, ks2, ki2 = gpu_ctx.score_cross(env, env, a_first, n_a, b_first, n_b, skip_self=skip_self, scores=False, k=k)
    assert np.array_equal(ki2, ki) and np.array_equal(ks2.view(np.uint64), ks.view(np.uint64))
    env.close(); st.close()


@pytest.mark.parametrize("route", ["tiles", "pairs"])
def test_chunks_forced_by_the_row_hook_change_nothing(gpu_ctx, oracle_mod, clouds, monkeypatch, route):
    _, members = clouds
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    if route == "pairs":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, members, ANCH_A)
    one = gpu_ctx.score_cross(env, env, 1, 38, 0, 42, skip_self=True, k=9)
    monkeypatch.setenv("LOCOHD_CROSS_ROWS", "4")
    launches = gpu_ctx.launch_count
    many = gpu_ctx.score_cross(env, env, 1, 38, 0, 42, skip_self=True, k=9)
    assert gpu_ctx.launch_count - launches >= 10   # 10 chunks of 4 rows
    for x, y in zip(one, many):
        assert np.array_equal(x.view(np.uint64) if x.dtype == np.float64 else x,
                              y.view(np.uint64) if y.dtype == np.float64 else y)
    env.close(); st.close()


def test_budget_sized_matrix_in_chunks_equals_one_device_chunk(gpu_ctx, oracle_mod):
    """400 x 100 000 scores (320 MB) in host memory take two chunks of the 256 MB scratch; into a device matrix the
    call writes one chunk straight to it.  Both, and the k nearest of both, are equal bit for bit."""
    import torch

    base = synth.gen(51, 625, 8, 7)
    clouds = [synth.partner(base, 1.5, 900 + i) for i in range(20)]
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, np.arange(base.n, dtype=np.uint32))
    assert len(env) == 100_000
    tiles = gpu_ctx.tile_launches
    host, ks, ki = gpu_ctx.score_cross(env, env, 1000, 400, 0, 100_000, k=8)
    assert gpu_ctx.tile_launches - tiles == 2      # two chunks of the tile kernel
    dev = torch.empty((400, 100_000), dtype=torch.float64, device="cuda")
    dks = torch.empty((400, 8), dtype=torch.float64, device="cuda")
    dki = torch.empty((400, 8), dtype=torch.int32, device="cuda")
    tiles = gpu_ctx.tile_launches
    gpu_ctx.score_cross(env, env, 1000, 400, 0, 100_000, scores=dev.data_ptr(), k=8, knn_scores=dks.data_ptr(),
                        knn_index=dki.data_ptr())
    assert gpu_ctx.tile_launches - tiles == 1      # one chunk
    assert np.array_equal(host.view(np.uint64), dev.cpu().numpy().view(np.uint64))
    assert np.array_equal(ks.view(np.uint64), dks.cpu().numpy().view(np.uint64))
    assert np.array_equal(ki, dki.cpu().numpy().view(np.uint32))
    env.close(); st.close()


def test_error_statuses(gpu_ctx, oracle_mod, clouds, monkeypatch):
    from loco_hd_b200._capi import LocoHDError, UNKNOWN_CATEGORY

    _, members = clouds
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, members[:2], ANCH_A)
    st2, other = _sets(gpu_ctx, members[2:], ANCH_B)
    n = len(env)

    def status(**kw):
        args = dict(a=env, b=env, a_first=0, n_a=4, b_first=0, n_b=8)
        args.update(kw)
        with pytest.raises(LocoHDError) as e:
            gpu_ctx.score_cross(**args)
        return e.value.status

    assert status(a_first=n - 3, n_a=4) == 8
    assert status(b_first=n + 1, n_b=0) == 8
    assert status(n_b=n + 1) == 8
    assert status(scores=False) == 10                                   # no output
    assert status(k=33) == 10
    assert status(k=8, skip_self=True) == 10                            # 7 columns left besides the rows' own
    gpu_ctx.score_cross(env, env, 0, 4, 0, 8, k=8)                      # without skip_self all 8 are eligible
    gpu_ctx.score_cross(env, env, 0, 4, 8, 8, skip_self=True, k=8)      # the rows' own columns lie outside the range
    assert status(b=other, skip_self=True, k=1) == 10
    with pytest.raises(LocoHDError, match="weight function index") as e:
        gpu_ctx.score_cross(env, env, 0, 4, 0, 8, wf_idx=1)
    assert e.value.status == 10
    # an unknown category inside an environment: the device error word, on either route
    bad = synth.partner(members[0], 0.5, 77)
    bad.cat = bad.cat.copy()
    bad.cat[ANCH_A[2] + 1] = UNKNOWN_CATEGORY
    st3, env3 = _sets(gpu_ctx, [bad], ANCH_A)
    for no_tiles in ("0", "1"):
        monkeypatch.setenv("LOCOHD_NO_TILES", no_tiles)
        with pytest.raises(LocoHDError) as e:
            gpu_ctx.score_cross(env3, env, 0, len(env3), 0, 8, k=2)
        assert e.value.status == 3
    for e in (env, other, env3, st, st2, st3):
        e.close()


def test_public_methods_equal_the_c_abi(gpu_ctx, oracle_mod, clouds):
    """LoCoHD.score_matrix / nearest_environments / score_pairs on the public class equal the C-ABI calls on the same
    environments; bad ranges, k and weight-function indices raise ValueError."""
    import loco_hd

    _, members = clouds
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, members, ANCH_A)
    lchd = loco_hd.LoCoHD([f"T{i}" for i in range(7)], loco_hd.WeightFunction("uniform", [3.0, 10.0]),
                          loco_hd.TagPairingRule({"accept_same": False}))
    offs = np.cumsum([0] + [c.n for c in members]).astype(np.uint64)
    pst = lchd.structures(offs, np.concatenate([c.xyz for c in members]), np.concatenate([c.cat for c in members]),
                          np.concatenate([c.tag for c in members]))
    penv = lchd.environments(pst, np.tile(ANCH_A, len(members)), THR,
                             anchor_struct=np.repeat(np.arange(len(members), dtype=np.uint32), len(ANCH_A)))
    M = lchd.score_matrix(penv, penv, (3, 30), (1, 40))
    want, _, _ = gpu_ctx.score_cross(env, env, 3, 27, 1, 39)
    assert np.array_equal(M, want)
    assert np.array_equal(lchd.score_matrix(penv, penv), gpu_ctx.score_cross(env, env)[0])
    ks, ki = lchd.nearest_environments(penv, penv, 6, a_range=(0, 20), exclude_self=True)
    _, wks, wki = gpu_ctx.score_cross(env, env, 0, 20, 0, len(env), skip_self=True, k=6)
    assert ki.dtype == np.uint32 and np.array_equal(ki, wki) and np.array_equal(ks, wks)
    pairs = np.array([[0, 5], [17, 2], [41, 41]], np.uint32)
    assert np.array_equal(lchd.score_pairs(penv, penv, pairs), gpu_ctx.score_pairs(env, env, pairs))
    for bad in [dict(a_range=(-1, 3)), dict(a_range=(5, 4)), dict(b_range=(0, len(env) + 1)), dict(wf_idx=1),
                dict(wf_idx=-1)]:
        with pytest.raises(ValueError):
            lchd.score_matrix(penv, penv, **bad)
    for k, kw in [(0, {}), (33, {}), (len(env), dict(exclude_self=True))]:
        with pytest.raises(ValueError):
            lchd.nearest_environments(penv, penv, k, **kw)
    with pytest.raises(ValueError):
        lchd.score_pairs(penv, penv, np.array([[0, len(env)]]))
    with pytest.raises(ValueError):
        lchd.score_pairs(penv, penv, np.array([[-1, 0]]))
    for e in (penv, pst, env, st):
        e.close()
