"""locohd_score_condensed: every unordered pair (i < j) of one range of one env-set once, in scipy's pdist order.  The
vector is checked against the CPU oracle on the anchor pairs it stands for (1e-9), bit for bit against the strict
upper triangle of locohd_score_cross on the same range and, on the pair route, against locohd_score_pairs on the
i < j list; chunked calls against one-chunk calls and a host output in several chunks against one launch into device
memory (bit for bit); squareform of the vector against both triangles of the matrix (the symmetry the call relies
on); and the error statuses and the public LoCoHD method.
"""
import numpy as np
import pytest

from benchdata import synth
from helpers import assert_scores_close, set_both

pytestmark = pytest.mark.gpu

THR = 10.0
ANCH = np.arange(0, 320, 23, dtype=np.uint32)   # 14 anchors per cloud


def _sets(ctx, clouds, anchors):
    """One structure set of `clouds`; environment e = anchor anchors[e % n] of cloud e // n."""
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    st = ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]), np.concatenate([c.cat for c in clouds]),
                            np.concatenate([c.tag for c in clouds]))
    anchors = np.asarray(anchors, np.uint32)
    env = ctx.envset_build(st, np.tile(anchors, len(clouds)), THR,
                           anchor_struct=np.repeat(np.arange(len(clouds), dtype=np.uint32), len(anchors)))
    return st, env


def _upper(M):
    """Strict upper triangle, row by row: the order of scipy.spatial.distance.pdist / squareform."""
    return M[np.triu_indices(M.shape[0], 1)]


def _pair_list(first, n):
    i, j = np.triu_indices(n, 1)
    return np.stack([i + first, j + first], axis=1).astype(np.uint32)


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint64)


@pytest.fixture(scope="module")
def clouds():
    base = synth.gen(31, 40, 8, 7)
    return [synth.partner(base, 1.5, 700 + i) for i in range(3)]


@pytest.mark.parametrize("first,n", [(3, 37), (0, 2), (10, 4), (7, 5), (0, 42)])
def test_vector_equals_the_oracle(gpu_ctx, oracle_mod, clouds, first, n):
    """Ranges that start inside the set with n no multiple of 4 (diagonal blocks with rows past the range), and the
    smallest ranges: every entry against the oracle's score of its anchor pair."""
    op = set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, ANCH)
    c = gpu_ctx.score_condensed(env, first, n)
    assert c.shape == (n * (n - 1) // 2,)
    pairs = _pair_list(first, n).astype(np.int64)
    want = np.empty(len(c))
    side = pairs // len(ANCH)
    for sa, sb in {(a, b) for a, b in side}:   # one oracle call per pair of clouds
        k = np.flatnonzero((side[:, 0] == sa) & (side[:, 1] == sb))
        ca, cb = clouds[sa], clouds[sb]
        want[k] = oracle_mod.from_primitives(op, ca.xyz, ca.cat, ca.tag, cb.xyz, cb.cat, cb.tag,
                                             ANCH[pairs[k] % len(ANCH)].astype(np.uint32), THR)
    assert_scores_close(c, want)
    env.close(); st.close()


def test_tile_route_equals_the_cross_matrix_bit_for_bit(gpu_ctx, oracle_mod, clouds):
    """W-keyed sets, Hellinger-2, unit weights: the tile kernel (counted by tile_launches) writes exactly the strict
    upper triangle of score_cross on the same range, on the same route."""
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, ANCH)
    for first, n in [(2, 37), (0, 42), (5, 8)]:
        before = gpu_ctx.tile_launches
        c = gpu_ctx.score_condensed(env, first, n)
        assert gpu_ctx.tile_launches - before == 1
        M, _, _ = gpu_ctx.score_cross(env, env, first, n, first, n)
        assert np.array_equal(_bits(c), _bits(_upper(M)))
    env.close(); st.close()


PAIR_ROUTE = {
    "no_tiles": dict(n_categories=7),
    "category_weights": dict(n_categories=7, category_weights=np.linspace(0.5, 2.0, 7)),
    "kolmogorov_smirnov": dict(n_categories=7, statistical_distance=("Kolmogorov-Smirnov", ())),
    "hellinger_3": dict(n_categories=7, statistical_distance=("Hellinger", (3.0,))),
    "c20": dict(n_categories=20),
    "wf_dict": dict(n_categories=7, weight_functions=(("uniform", (3.0, 10.0)), ("kumaraswamy", (2.0, 9.0, 2.0, 3.0)))),
}


@pytest.mark.parametrize("case", sorted(PAIR_ROUTE))
def test_pair_route_equals_cross_and_score_pairs_bit_for_bit(gpu_ctx, oracle_mod, monkeypatch, case):
    """Configurations the tile kernel does not take (and LOCOHD_NO_TILES): explicit pairs on the pair kernel, the
    same kernel and arithmetic as score_cross and score_pairs, so all three agree bit for bit."""
    kw = dict(PAIR_ROUTE[case])
    C = kw.pop("n_categories")
    base = synth.gen(41, 40, 8, C)
    members = [synth.partner(base, 1.5, 800 + i) for i in range(2)]
    set_both(gpu_ctx, oracle_mod, C, tag_rule={"accept_same": False}, **kw)
    if case == "no_tiles":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, members, ANCH)
    wf = 1 if case == "wf_dict" else 0
    first, n = 1, 25
    before = gpu_ctx.tile_launches
    c = gpu_ctx.score_condensed(env, first, n, wf_idx=wf)
    M, _, _ = gpu_ctx.score_cross(env, env, first, n, first, n, wf_idx=wf)
    pairs = _pair_list(first, n)
    ref = gpu_ctx.score_pairs(env, env, pairs, wf_idx=np.full(len(pairs), wf, np.uint32))
    assert gpu_ctx.tile_launches == before
    assert np.array_equal(_bits(c), _bits(_upper(M)))
    assert np.array_equal(_bits(c), _bits(ref))
    env.close(); st.close()


@pytest.mark.parametrize("route", ["tiles", "pairs"])
def test_squareform_is_both_triangles_of_the_matrix(gpu_ctx, oracle_mod, clouds, monkeypatch, route):
    """Hellinger is symmetric in its two environments: the lower triangle of score_matrix, scored with the roles
    swapped, is the vector too (1e-12), so clustering on the vector clusters on the matrix."""
    from scipy.spatial.distance import squareform

    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    if route == "pairs":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, clouds, ANCH)
    c = gpu_ctx.score_condensed(env, 3, 37)
    M, _, _ = gpu_ctx.score_cross(env, env, 3, 37, 3, 37)
    S = squareform(c)
    off = ~np.eye(37, dtype=bool)
    assert np.abs(S - M)[off].max() <= 1e-12
    assert np.abs(S - M.T)[off].max() <= 1e-12
    env.close(); st.close()


@pytest.mark.parametrize("route", ["tiles", "pairs"])
def test_chunks_forced_by_the_row_hook_change_nothing(gpu_ctx, oracle_mod, clouds, monkeypatch, route):
    """LOCOHD_CROSS_ROWS=4: one chunk per row block.  38 rows from environment 1 are 10 row blocks, 10 chunks; with 37
    rows the last block holds only the last row, which has no pair, and is not launched."""
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    if route == "pairs":
        monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    st, env = _sets(gpu_ctx, clouds, ANCH)
    for n, chunks in [(38, 10), (37, 9)]:
        monkeypatch.delenv("LOCOHD_CROSS_ROWS", raising=False)
        one = gpu_ctx.score_condensed(env, 1, n)
        monkeypatch.setenv("LOCOHD_CROSS_ROWS", "4")
        launches, tiles = gpu_ctx.launch_count, gpu_ctx.tile_launches
        many = gpu_ctx.score_condensed(env, 1, n)
        if route == "tiles":
            assert gpu_ctx.tile_launches - tiles == chunks
        else:
            assert gpu_ctx.tile_launches == tiles
            assert gpu_ctx.launch_count - launches >= 2 * chunks   # pair list and pair kernel per chunk
        assert np.array_equal(_bits(one), _bits(many))
    env.close(); st.close()


def test_budget_sized_vector_in_chunks_equals_one_device_launch(gpu_ctx, oracle_mod):
    """12 000 environments: 71 994 000 scores (576 MB) into host memory take three chunks of the 256 MB scratch (807,
    1 409 and 784 row blocks - later chunks take more of the shorter rows); into a torch device buffer the call writes
    the whole triangle with one launch.  Both are equal bit for bit."""
    import torch

    base = synth.gen(51, 500, 8, 7)
    clouds = [synth.partner(base, 1.5, 900 + i) for i in range(3)]
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, np.arange(base.n, dtype=np.uint32))
    n = len(env)
    assert n == 12_000
    tiles = gpu_ctx.tile_launches
    host = gpu_ctx.score_condensed(env)
    assert gpu_ctx.tile_launches - tiles == 3
    dev = torch.empty(n * (n - 1) // 2, dtype=torch.float64, device="cuda")
    tiles = gpu_ctx.tile_launches
    gpu_ctx.score_condensed(env, out=dev.data_ptr())
    assert gpu_ctx.tile_launches - tiles == 1
    assert np.array_equal(_bits(host), dev.cpu().numpy().view(np.uint64))
    env.close(); st.close()


def test_error_statuses(gpu_ctx, oracle_mod, clouds, monkeypatch):
    from loco_hd_b200._capi import LocoHDError, UNKNOWN_CATEGORY

    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, ANCH)
    n = len(env)

    def status(*args, **kw):
        with pytest.raises(LocoHDError) as e:
            gpu_ctx.score_condensed(env, *args, **kw)
        return e.value.status

    assert status(n - 3, 4) == 8
    assert status(n + 1, 0) == 8
    assert status(0, n + 1) == 8
    assert status(0, 4, out=0) == 10                                    # no output
    with pytest.raises(LocoHDError, match="weight function index") as e:
        gpu_ctx.score_condensed(env, 0, 8, wf_idx=1)
    assert e.value.status == 10
    # n < 2: nothing to score, no launch, no output needed
    launches = gpu_ctx.launch_count
    for first, m in [(0, 0), (5, 1), (n, 0)]:
        assert gpu_ctx.score_condensed(env, first, m).shape == (0,)
        gpu_ctx.score_condensed(env, first, m, out=0)
    assert gpu_ctx.launch_count == launches
    # asymmetric statistical distances: one triangle would not stand for the matrix
    for sd in [("Kullback-Leibler", (1e-6,)), ("Renyi", (1.7, 0.2))]:
        set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False}, statistical_distance=sd)
        st2, env2 = _sets(gpu_ctx, clouds[:1], ANCH)
        with pytest.raises(LocoHDError, match="locohd_score_cross") as e:
            gpu_ctx.score_condensed(env2, 0, 8)
        assert e.value.status == 10
        env2.close(); st2.close()
    # an unknown category inside an environment: the device error word, on either route
    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    bad = synth.partner(clouds[0], 0.5, 77)
    bad.cat = bad.cat.copy()
    bad.cat[ANCH[2] + 1] = UNKNOWN_CATEGORY
    st3, env3 = _sets(gpu_ctx, [clouds[1], bad], ANCH)
    for no_tiles in ("0", "1"):
        monkeypatch.setenv("LOCOHD_NO_TILES", no_tiles)
        tiles = gpu_ctx.tile_launches
        with pytest.raises(LocoHDError) as e:
            gpu_ctx.score_condensed(env3)
        assert e.value.status == 3
        assert (gpu_ctx.tile_launches > tiles) == (no_tiles == "0")
    for e in (env, env3, st, st3):
        e.close()


def test_public_method_equals_the_c_abi(gpu_ctx, oracle_mod, clouds):
    """LoCoHD.score_condensed on the public class equals the C-ABI call on the same environments and feeds scipy's
    clustering; bad ranges, weight-function indices and an asymmetric distance raise ValueError."""
    import loco_hd
    from scipy.cluster.hierarchy import linkage

    set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    st, env = _sets(gpu_ctx, clouds, ANCH)
    cats = [f"T{i}" for i in range(7)]
    lchd = loco_hd.LoCoHD(cats, loco_hd.WeightFunction("uniform", [3.0, 10.0]),
                          loco_hd.TagPairingRule({"accept_same": False}))
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    xyz, cat, tag = (np.concatenate([getattr(c, f) for c in clouds]) for f in ("xyz", "cat", "tag"))
    pst = lchd.structures(offs, xyz, cat, tag)
    penv = lchd.environments(pst, np.tile(ANCH, len(clouds)), THR,
                             anchor_struct=np.repeat(np.arange(len(clouds), dtype=np.uint32), len(ANCH)))
    c = lchd.score_condensed(penv, (3, 30))
    assert np.array_equal(_bits(c), _bits(gpu_ctx.score_condensed(env, 3, 27)))
    assert np.array_equal(_bits(lchd.score_condensed(penv)), _bits(gpu_ctx.score_condensed(env)))
    assert lchd.score_condensed(penv, (4, 5)).shape == (0,)
    assert linkage(lchd.score_condensed(penv), "average").shape == (len(env) - 1, 4)
    for bad in [dict(env_range=(-1, 3)), dict(env_range=(5, 4)), dict(env_range=(0, len(env) + 1)), dict(wf_idx=1),
                dict(wf_idx=-1)]:
        with pytest.raises(ValueError):
            lchd.score_condensed(penv, **bad)
    kl = loco_hd.LoCoHD(cats, loco_hd.WeightFunction("uniform", [3.0, 10.0]),
                        loco_hd.TagPairingRule({"accept_same": False}),
                        statistical_distance=loco_hd.StatisticalDistance("Kullback-Leibler", [1e-6]))
    kst = kl.structures(offs, xyz, cat, tag)
    kenv = kl.environments(kst, np.tile(ANCH, len(clouds)), THR,
                           anchor_struct=np.repeat(np.arange(len(clouds), dtype=np.uint32), len(ANCH)))
    with pytest.raises(ValueError, match="symmetric"):
        kl.score_condensed(kenv)
    for e in (penv, pst, kenv, kst, env, st):
        e.close()
