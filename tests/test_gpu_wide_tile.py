"""score_wide_kernel: job lists that fill 32 x 32 tiles to at least 80 % (the all-vs-all ensemble of 1000 members)
are scored one CTA per (tile, anchor), one lane per anchor pair walking the whole merged list from the two anchors.
Every case
asserts that the wide kernel ran (locohd_ctx_wide_launches) and checks the scores against the CPU oracle (1e-9); the
4 x 4 tile kernel (LOCOHD_WIDE_TILES=0) and the one-pair-per-warp kernel (LOCOHD_NO_TILES=1) score the same jobs
within 1e-12 (same arithmetic, other points where D and R are rebuilt).  A lane's walk does not depend on which
unit order, run length or table replication the launch uses, so those switches must not change a bit.
"""
import numpy as np
import pytest

from benchdata import synth
from helpers import SCORE_TOL, assert_scores_close, set_both
from loco_hd_b200 import _capi, batch

pytestmark = pytest.mark.gpu

JOB = [("a_first", "<u8"), ("b_first", "<u8"), ("n", "<u8")]
OTHERS = {"accept_same": False}


def _resident(ctx, clouds, anchors, threshold):
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    st = ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]), np.concatenate([c.cat for c in clouds]),
                            np.concatenate([c.tag for c in clouds]))
    a_struct = np.repeat(np.arange(len(clouds), dtype=np.uint32), len(anchors))
    env = ctx.envset_build(st, np.tile(np.asarray(anchors, np.uint32), len(clouds)), threshold, anchor_struct=a_struct)
    return st, env


def _jobs(pairs, n):
    return np.array([(i * n, j * n, n) for i, j in pairs], dtype=JOB)


def _grid_pairs(n_a, n_b):
    """All (i, j) of two environment sets, in 4 x 4 blocks."""
    return np.array([(i, j) for bi in range(0, n_a, 4) for bj in range(0, n_b, 4)
                     for i in range(bi, min(bi + 4, n_a)) for j in range(bj, min(bj + 4, n_b))], dtype=np.int64)


def _score(ctx, env_a, env_b, jobs, route="wide", **kw):
    """Scores of one call and the route it took: 'wide', 'tile' (4 x 4) or 'pair'."""
    tiles, wide = ctx.tile_launches, ctx.wide_launches
    res = ctx.score_jobs_stats(env_a, env_b, jobs, scores=True, **kw)
    took = "wide" if ctx.wide_launches > wide else "tile" if ctx.tile_launches > tiles else "pair"
    assert took == route, f"expected the {route} route, took {took}"
    return res


def _three_routes(ctx, monkeypatch, env_a, env_b, jobs, **kw):
    wide = _score(ctx, env_a, env_b, jobs, "wide", **kw)
    with monkeypatch.context() as m:
        m.setenv("LOCOHD_WIDE_TILES", "0")
        tile = _score(ctx, env_a, env_b, jobs, "tile", **kw)
    with monkeypatch.context() as m:
        m.setenv("LOCOHD_NO_TILES", "1")
        pair = _score(ctx, env_a, env_b, jobs, "pair", **kw)
    assert np.abs(wide["scores"] - tile["scores"]).max() <= 1e-12
    assert np.abs(wide["scores"] - pair["scores"]).max() <= 1e-12
    return wide


def _oracle(oracle_mod, op, clouds_a, clouds_b, pairs, anchors_a, anchors_b, threshold):
    an = np.stack([anchors_a, anchors_b], axis=1).astype(np.uint32)
    out = np.empty((len(pairs), len(anchors_a)))
    for k, (i, j) in enumerate(np.asarray(pairs).tolist()):
        a, b = clouds_a[i], clouds_b[j]
        out[k] = oracle_mod.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, an, threshold)
    return out


def test_ensemble_of_160_members_in_blocked_order(gpu_ctx, oracle_mod, monkeypatch):
    """160 members in batch.blocked_pairs order: fifteen 32 x 32 tiles filled to 83 %, five of them diagonal blocks
    (the cells on and below the diagonal are absent), member 40 an exact copy of member 9.  Unit order, run length and
    the unreplicated table instantiation change no bit; job means, anchor means and stds follow the scores."""
    base = synth.gen(61, 6, 4, 7)
    members = [synth.partner(base, 1.5, 1600 + i) for i in range(160)]
    members[40] = members[9]
    anchors = np.arange(base.n, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0))], tag_rule=OTHERS)
    st, env = _resident(gpu_ctx, members, anchors, 10.0)
    pairs = batch.blocked_pairs(160, 4)
    jobs = _jobs(pairs, base.n)
    kw = dict(job_means=True, anchor_means=True, anchor_stds=True)
    got = _three_routes(gpu_ctx, monkeypatch, env, env, jobs, **kw)
    want = _oracle(oracle_mod, op, members, members, pairs, anchors, anchors, 10.0)
    assert_scores_close(got["scores"], want.ravel())
    k = [tuple(p) for p in pairs.tolist()].index((9, 40))
    assert np.all(got["scores"].reshape(len(pairs), base.n)[k] == 0.0), "identical members score exactly 0"
    assert np.abs(got["job_means"] - want.mean(axis=1)).max() <= SCORE_TOL
    assert np.abs(got["anchor_means"] - want.mean(axis=0)).max() <= SCORE_TOL
    assert np.abs(got["anchor_stds"] - want.std(axis=0)).max() <= SCORE_TOL
    for name, value in (("LOCOHD_TILE_SLICE", "0"), ("LOCOHD_TILE_SLICE", "8"), ("LOCOHD_TILE_SLICE", "40"),
                        ("LOCOHD_TILE_RUN", "1"), ("LOCOHD_TILE_RUN", "3"), ("LOCOHD_TILE_REP", "0")):
        with monkeypatch.context() as m:
            m.setenv(name, value)
            other = _score(gpu_ctx, env, env, jobs, "wide", job_means=True)
        assert np.array_equal(other["scores"], got["scores"]), f"{name}={value}"
        assert np.array_equal(other["job_means"], got["job_means"]), f"{name}={value}"
    env.close(); st.close()


def test_partial_tiles_of_two_sets_and_a_contiguous_share(gpu_ctx, oracle_mod, monkeypatch):
    """Rows from 60 structures, columns from 32 others (12 categories: 16 count rows per lane): a full and a partial
    tile row.  The second half of the list (what rank 1 of 2 scores) starts inside the first tile and is regrouped into
    one partial tile of 30 rows; its scores are those of the whole list, bit for bit."""
    base_a = synth.gen(62, 10, 4, 12)
    base_b = synth.gen(63, 9, 4, 12)
    rows = [synth.partner(base_a, 1.5, 1700 + i) for i in range(60)]
    cols = [synth.partner(base_b, 1.5, 1800 + i) for i in range(32)]
    n = min(base_a.n, base_b.n)
    an = np.arange(n, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 12, [("uniform", (3.0, 10.0))], tag_rule=OTHERS)
    st_a, env_a = _resident(gpu_ctx, rows, an, 10.0)
    st_b, env_b = _resident(gpu_ctx, cols, an, 10.0)
    pairs = _grid_pairs(60, 32)
    jobs = _jobs(pairs, n)
    got = _three_routes(gpu_ctx, monkeypatch, env_a, env_b, jobs, job_means=True)
    want = _oracle(oracle_mod, op, rows, cols, pairs, an, an, 10.0)
    assert_scores_close(got["scores"], want.ravel())
    sl = batch.contiguous_share(len(jobs), 1, 2)
    part = _score(gpu_ctx, env_a, env_b, jobs[sl], "wide")
    assert np.array_equal(part["scores"], got["scores"].reshape(len(pairs), n)[sl].ravel())
    for h in (env_a, env_b, st_a, st_b):
        h.close()


def _copies_32(ctx, oracle_mod, monkeypatch, op, a, b, an_a, an_b, threshold):
    """32 copies of cloud a as rows against 32 copies of cloud b as columns: one full wide tile of the same pair."""
    st_a, env_a = _resident(ctx, [a] * 32, an_a, threshold)
    st_b, env_b = _resident(ctx, [b] * 32, an_b, threshold)
    pairs = _grid_pairs(32, 32)
    got = _three_routes(ctx, monkeypatch, env_a, env_b, _jobs(pairs, len(an_a)))["scores"].reshape(1024, len(an_a))
    want = _oracle(oracle_mod, op, [a], [b], [(0, 0)], an_a, an_b, threshold)[0]
    assert_scores_close(got.ravel(), np.tile(want, 1024))
    assert np.all(got == got[0]), "the 1024 cells of the tile hold the same pair of structures"
    for h in (env_a, env_b, st_a, st_b):
        h.close()
    return got[0]


def test_compositions_identical_then_different_on_a_wide_tile(gpu_ctx, oracle_mod, monkeypatch):
    """As in test_gpu_tile_walk: B is A scaled by 1 + 1e-6, so the walk alternates identical (H exactly 0) and
    differing compositions on every event."""
    a = synth.gen(41, 40, 8, 7)
    b = synth.Cloud(np.ascontiguousarray(a.xyz * (1.0 + 1e-6)), a.cat.copy(), a.tag.copy(), a.k, a.centroid_cat)
    anchors = np.arange(0, a.n, 5, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (0.0, 10.0))], tag_rule=OTHERS)
    got = _copies_32(gpu_ctx, oracle_mod, monkeypatch, op, a, b, anchors, anchors, 10.0)
    assert 0.0 < got.min() and got.max() < 0.1


def test_small_h2_runs_and_last_event_on_a_wide_tile(gpu_ctx, oracle_mod, monkeypatch):
    """As in test_gpu_tile_walk: runs of category-0 events keep H^2 a rounding residue, other categories break them,
    and the complete compositions are proportional (the last event ends in the difference form).  Walks of 448
    events: D and R are rebuilt from the counts three times inside them."""
    rng = np.random.default_rng(91)
    n_points = 150
    direction = rng.normal(size=(n_points, 3))
    direction /= np.linalg.norm(direction, axis=1, keepdims=True)
    xyz_a = direction * (8.0 * rng.random(n_points) ** (1.0 / 3.0))[:, None]
    cat_a = np.where(rng.random(n_points) < 0.9, 0, rng.integers(1, 3, n_points)).astype(np.uint16)
    xyz_b = np.repeat(xyz_a, 2, axis=0)
    xyz_b[1::2, 0] += 1e-7
    cat_b = np.repeat(cat_a, 2)
    a = synth.Cloud(xyz_a, cat_a, np.arange(n_points, dtype=np.uint32), 1)
    b = synth.Cloud(xyz_b, cat_b, np.arange(2 * n_points, dtype=np.uint32) + n_points, 1)
    an_a = np.arange(0, n_points, 10, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 3, [("uniform", (0.0, 30.0))], tag_rule=OTHERS)
    got = _copies_32(gpu_ctx, oracle_mod, monkeypatch, op, a, b, an_a, 2 * an_a, 20.0)
    assert got.max() < 0.2


def _ball(seed, n, C, radius):
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    xyz = d * (radius * rng.random(n) ** (1.0 / 3.0))[:, None]
    return synth.Cloud(xyz, rng.permutation(np.arange(n) % C).astype(np.uint16), np.arange(n, dtype=np.uint32), 1)


@pytest.mark.parametrize("members,route", [(367, "wide"), (368, "tile")])
def test_largest_environments_the_stage_takes(gpu_ctx, oracle_mod, monkeypatch, members, route):
    """Balls of `members` points inside the threshold: every environment holds them all.  367 members (C <= 8) are
    the largest whose 64 staged environments, count rows and tables fit 227 KB; one more takes the 4 x 4 tiles.  A
    walk of 732 events rebuilds D and R five times."""
    a = _ball(71, members, 7, 4.9)
    b = synth.Cloud(a.xyz + np.random.default_rng(72).normal(scale=0.02, size=a.xyz.shape), a.cat[::-1].copy(),
                    a.tag.copy(), 1)
    b.xyz *= 4.9 / max(4.9, np.linalg.norm(b.xyz, axis=1).max())
    an = np.arange(0, members, 61, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (0.0, 10.0))], tag_rule=OTHERS)
    st_a, env_a = _resident(gpu_ctx, [a] * 32, an, 10.0)
    st_b, env_b = _resident(gpu_ctx, [b] * 32, an, 10.0)
    for env in (env_a, env_b):
        off = np.empty(len(env) + 1, np.uint64)
        gpu_ctx._check(gpu_ctx.lib.locohd_envset_dump(gpu_ctx.h, env.h, _capi._p(off), None, None, None))
        assert np.all(np.diff(off.astype(np.int64)) == members)
    jobs = _jobs(_grid_pairs(32, 32), len(an))
    got = _score(gpu_ctx, env_a, env_b, jobs, route)["scores"].reshape(1024, len(an))
    want = _oracle(oracle_mod, op, [a], [b], [(0, 0)], an, an, 10.0)[0]
    assert_scores_close(got.ravel(), np.tile(want, 1024))
    assert got.min() > 0.0
    for h in (env_a, env_b, st_a, st_b):
        h.close()


def test_wide_tiles_report_unknown_categories(gpu_ctx, oracle_mod):
    """pmf.rs:38-42: a primitive type the instance does not know is an error once it is met inside an environment;
    the wide kernel finds it in the staged environments before any walk."""
    from loco_hd_b200._capi import LocoHDError, UNKNOWN_CATEGORY
    base = synth.gen(64, 8, 4, 7)
    members = [synth.partner(base, 1.0, 1900 + i) for i in range(32)]
    members[25].cat[11] = UNKNOWN_CATEGORY
    anchors = np.arange(base.n, dtype=np.uint32)
    set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0))], tag_rule=OTHERS)
    st, env = _resident(gpu_ctx, members, anchors, 10.0)
    wide = gpu_ctx.wide_launches
    with pytest.raises(LocoHDError) as ei:
        gpu_ctx.score_jobs_stats(env, env, _jobs(_grid_pairs(32, 32), base.n), scores=True)
    assert ei.value.status == 3 and gpu_ctx.wide_launches > wide
    env.close(); st.close()
