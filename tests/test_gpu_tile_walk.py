"""The per-event walk of score_tile_kernel on the cases its bookkeeping has to get right: compositions that become
identical inside a lane's chunk and differ again on the next event (the exact 0 comes from sum_r |a_r - b_r|, kept
by +-1 per event), H^2 falling below and rising above 1e-8 on consecutive events of one chunk (the difference form
from the counts takes over and hands back), and a walk whose last event ends in that branch (its H is the one the
tail to infinity uses).  Every case runs on a 4 x 4 tile of structure pairs (the tile kernel takes it) and is checked
against the CPU oracle (1e-9) and against the one-pair-per-warp kernel on the same jobs (1e-12).
"""
import numpy as np
import pytest

from benchdata import synth
from helpers import assert_scores_close, set_both

pytestmark = pytest.mark.gpu

JOB = [("a_first", "<u8"), ("b_first", "<u8"), ("n", "<u8")]


def _resident(ctx, cloud, anchors, threshold, copies=4):
    offs = np.arange(copies + 1, dtype=np.uint64) * np.uint64(cloud.n)
    st = ctx.structs_create(offs, np.concatenate([cloud.xyz] * copies), np.concatenate([cloud.cat] * copies),
                            np.concatenate([cloud.tag] * copies))
    a_struct = np.repeat(np.arange(copies, dtype=np.uint32), len(anchors))
    env = ctx.envset_build(st, np.tile(np.asarray(anchors, np.uint32), copies), threshold, anchor_struct=a_struct)
    return st, env


def _tile_and_pair(ctx, monkeypatch, env_a, env_b, n):
    jobs = np.array([(i * n, j * n, n) for i in range(4) for j in range(4)], dtype=JOB)
    before = ctx.tile_launches
    tiled = ctx.score_jobs_stats(env_a, env_b, jobs, scores=True)["scores"]
    assert ctx.tile_launches > before, "the 4 x 4 tile takes the tile kernel"
    monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    before = ctx.tile_launches
    plain = ctx.score_jobs_stats(env_a, env_b, jobs, scores=True)["scores"]
    assert ctx.tile_launches == before
    monkeypatch.delenv("LOCOHD_NO_TILES")
    return tiled.reshape(16, n), plain.reshape(16, n)


def _check(ctx, oracle, monkeypatch, op, a, b, an_a, an_b, threshold):
    st_a, env_a = _resident(ctx, a, an_a, threshold)
    st_b, env_b = _resident(ctx, b, an_b, threshold)
    tiled, plain = _tile_and_pair(ctx, monkeypatch, env_a, env_b, len(an_a))
    an = np.stack([an_a, an_b], axis=1).astype(np.uint32)
    want = oracle.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, an, threshold)
    assert_scores_close(tiled.ravel(), np.tile(want, 16))
    assert np.all(tiled == tiled[0]), "the 16 cells of the tile hold the same pair of structures"
    assert np.abs(tiled - plain).max() <= 1e-12
    for h in (env_a, env_b, st_a, st_b):
        h.close()
    return tiled[0], want


def test_compositions_identical_inside_a_chunk_then_different(gpu_ctx, oracle_mod, monkeypatch):
    """B is A scaled by 1 + 1e-6: every distance of B is a hair longer than the same distance of A, so the merge walks
    a1 b1 a2 b2 ... - the compositions are identical after every B event and differ after every A event, dozens of
    times inside every lane's chunk."""
    a = synth.gen(41, 40, 8, 7)
    b = synth.Cloud(np.ascontiguousarray(a.xyz * (1.0 + 1e-6)), a.cat.copy(), a.tag.copy(), a.k, a.centroid_cat)
    anchors = np.arange(a.n, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (0.0, 10.0))], tag_rule={"accept_same": False})
    got, want = _check(gpu_ctx, oracle_mod, monkeypatch, op, a, b, anchors, anchors, 10.0)
    # H is exactly 0 on every other event and of order 1 / n on the rest: the scores are small but not 0
    assert 0.0 < got.min() and got.max() < 0.1


def test_small_h2_on_consecutive_events_and_on_the_last_event(gpu_ctx, oracle_mod, monkeypatch):
    """Nine in ten points of category 0: runs of category-0 events keep both compositions pure (proportional, H = 0,
    H^2 a rounding residue below 1e-8) for many consecutive events of a chunk, and each other category breaks the run
    (H^2 well above 1e-8 on the next event).  B holds every point of A twice, so the complete compositions are
    proportional too: the last event of every walk ends in the difference-form branch."""
    rng = np.random.default_rng(91)
    n_points = 300
    direction = rng.normal(size=(n_points, 3))
    direction /= np.linalg.norm(direction, axis=1, keepdims=True)
    xyz_a = direction * (8.0 * rng.random(n_points) ** (1.0 / 3.0))[:, None]
    cat_a = np.where(rng.random(n_points) < 0.9, 0, rng.integers(1, 3, n_points)).astype(np.uint16)
    xyz_b = np.repeat(xyz_a, 2, axis=0)
    xyz_b[1::2, 0] += 1e-7
    cat_b = np.repeat(cat_a, 2)
    a = synth.Cloud(xyz_a, cat_a, np.arange(n_points, dtype=np.uint32), 1)
    b = synth.Cloud(xyz_b, cat_b, np.arange(2 * n_points, dtype=np.uint32) + n_points, 1)
    an_a = np.arange(0, n_points, 2, dtype=np.uint32)
    an_b = 2 * an_a
    op = set_both(gpu_ctx, oracle_mod, 3, [("uniform", (0.0, 30.0))], tag_rule={"accept_same": False})
    got, _ = _check(gpu_ctx, oracle_mod, monkeypatch, op, a, b, an_a, an_b, 20.0)
    assert got.max() < 0.2
