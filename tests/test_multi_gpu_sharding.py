"""The N > 1 path: jobs are dealt to ranks, every rank scores its share, results are assembled on the host — no
collective on the scoring path.  CPU: the dealing/assembling logic alone and under a world_size-2 gloo group.
GPU: the sharded all-vs-all ensemble equals the unsharded one and the oracle."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from benchdata import synth
from loco_hd_b200 import batch

ROOT = Path(__file__).resolve().parent.parent


def test_deal_jobs_is_balanced_and_complete():
    rng = np.random.default_rng(1)
    for world in (1, 2, 3, 8):
        sizes = rng.integers(1, 10000, size=257)
        shares = batch.deal_jobs(sizes, world)
        assert len(shares) == world
        assert np.array_equal(np.sort(np.concatenate(shares)), np.arange(len(sizes)))
        loads = np.array([sizes[s].sum() for s in shares])
        assert loads.max() - loads.min() <= sizes.max()
    assert [len(s) for s in batch.deal_jobs([5, 5, 5, 5], 2)] == [2, 2]
    assert batch.deal_jobs([], 4)[0].size == 0


def test_all_pairs_and_assemble():
    pairs = batch.all_pairs(5)
    assert len(pairs) == 10 and all(i < j for i, j in pairs)
    ids = [np.array([0, 3]), np.array([1, 2])]
    vals = [np.array([10.0, 13.0]), np.array([11.0, 12.0])]
    assert np.array_equal(batch.assemble(ids, vals, 4), [10.0, 11.0, 12.0, 13.0])


def test_world_size_2_gloo(tmp_path):
    out = tmp_path / "ok.txt"
    env = dict(os.environ, LOCOHD_TEST_OUT=str(out), MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29533", str(ROOT / "tests" / "_dist_worker.py")]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    assert out.read_text() == "ok"


@pytest.mark.gpu
def test_sharded_ensemble_matches_unsharded_and_oracle(gpu_ctx, oracle_mod):
    base = synth.gen(9, 40, 8, 7)
    clouds = [synth.config5_member(base, i) for i in range(6)]
    anchors = np.arange(base.n, dtype=np.uint32)
    gpu_ctx.set_params(7, [("uniform", (3.0, 10.0))], tag_rule={"accept_same": False})
    whole = batch.ensemble_all_vs_all(gpu_ctx, clouds, anchors, 10.0)
    parts = [batch.ensemble_all_vs_all(gpu_ctx, clouds, anchors, 10.0, rank=r, world=3, gather=False) for r in range(3)]
    merged = np.where(np.isnan(parts[0]), np.where(np.isnan(parts[1]), parts[2], parts[1]), parts[0])
    assert np.array_equal(merged, whole)
    # per-atom statistics over all structure pairs, pooled over chunks of pairs (compare_ensembles.py:299)
    ens = batch.ResidentEnsemble.build(gpu_ctx, clouds, anchors, 10.0)
    all_p = batch.all_pairs(len(clouds))
    m1, am1, as1 = ens.pair_means_and_anchor_stats(all_p)
    m2, am2, as2 = ens.pair_means_and_anchor_stats(all_p, chunk=4)
    jobs = ens.job_table(all_p)
    per_anchor = gpu_ctx.score_jobs(ens.env, ens.env, jobs).reshape(len(all_p), len(anchors))
    ens.close()
    assert np.array_equal(m1, whole) and np.array_equal(m2, whole)
    for am, asd in ((am1, as1), (am2, as2)):
        assert np.abs(am - per_anchor.mean(axis=0)).max() <= 1e-14 and np.abs(asd - per_anchor.std(axis=0)).max() <= 1e-14
    op = oracle_mod.Params(7, [("uniform", [3.0, 10.0])], tag_rule={"accept_same": False})
    pairs = batch.all_pairs(len(clouds))
    an = np.stack([anchors, anchors], axis=1)
    for k in (0, 7, 14):
        i, j = pairs[k]
        a, b = clouds[i], clouds[j]
        ref = oracle_mod.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, an, 10.0)
        assert abs(ref.mean() - whole[k]) <= 1e-9


def _load_bench():
    import importlib.util

    spec = importlib.util.spec_from_file_location("locohd_bench", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


def test_bench_ensemble_jobs_are_dealt_without_overlap():
    """bench.py's config-5 workload: the i < j structure pairs are dealt round-robin over the ranks (strong scaling,
    no collective), every pair exactly once, and the per-job event count used for the roofline equals the naive sum."""
    import types

    bench = _load_bench()
    args = types.SimpleNamespace(ensemble=7, pairs=2, models=3, frames=3)
    world = 3
    seen = []
    for rank in range(world):
        wl = bench.make_workload("cfg5", rank, world, args)
        assert wl.scaling == "strong" and wl.n_pairs == len(wl.jobs) * 5000
        seen += [tuple(g) for g in wl.job_groups]
        # sum of (Ma + Mb - 1) per job from environment offsets, as bench.py computes it, against the plain loop
        rng = np.random.default_rng(rank)
        sizes = rng.integers(1, 400, size=len(wl.anchor_prim)).astype(np.uint64)
        off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        ja, jb, jn = (wl.jobs[k].astype(np.int64) for k in ("a_first", "b_first", "n"))
        members = (off[ja + jn] - off[ja]).astype(np.int64) + (off[jb + jn] - off[jb]).astype(np.int64)
        naive = sum(int(sizes[j["a_first"]:j["a_first"] + j["n"]].sum() + sizes[j["b_first"]:j["b_first"] + j["n"]].sum())
                    for j in wl.jobs)
        assert int(members.sum()) == naive
    assert sorted(seen) == [(i, j) for i in range(7) for j in range(i + 1, 7)]


def test_blocked_pairs_and_contiguous_shares():
    """The L2-friendly job order holds every i < j pair once, tiles touch at most 2 * block structures, and the
    contiguous per-rank runs partition the list."""
    for n, block in ((1, 4), (2, 4), (7, 4), (33, 4), (20, 3)):
        order = batch.blocked_pairs(n, block)
        assert sorted(map(tuple, order.tolist())) == sorted(map(tuple, batch.all_pairs(n).tolist()))
        tiles = {}
        for k, (i, j) in enumerate(order.tolist()):
            tiles.setdefault((i // block, j // block), []).append(k)
        for ks in tiles.values():          # a tile's jobs are consecutive in the order
            assert ks == list(range(ks[0], ks[0] + len(ks)))
    n_jobs = 101
    for world in (1, 2, 3, 8):
        runs = [batch.contiguous_share(n_jobs, r, world) for r in range(world)]
        assert [x for s in runs for x in range(n_jobs)[s]] == list(range(n_jobs))
        assert max(s.stop - s.start for s in runs) - min(s.stop - s.start for s in runs) <= 1


def test_job_lists_group_into_tiles_on_the_host():
    """locohd_plan_job_tiles (no device): the all-vs-all ensemble of compare_ensembles.py:250-296 groups into 4 x 4
    tiles of structure pairs whatever the order of the list; one-against-many lists (trajectory_analyzer.py:112-120)
    and lists of unequal jobs do not."""
    from loco_hd_b200 import _capi

    n = 5000

    def jobs_of(pairs):
        return np.array([(i * n, j * n, n) for i, j in pairs], dtype=batch.JOB_DTYPE)

    S = 40                                            # 10 block rows: 45 full tiles + 10 diagonal ones
    blocked = batch.blocked_pairs(S, 4)
    plan = _capi.plan_job_tiles(jobs_of(blocked))
    assert plan["pays"] and plan["tiles"] == 55 and plan["rows"] == 45 * 4 + 10 * 3
    rng = np.random.default_rng(3)
    for order in (batch.all_pairs(S), blocked[rng.permutation(len(blocked))]):   # row-major, shuffled
        p2 = _capi.plan_job_tiles(jobs_of(order))
        # (ranked separately, the A runs are structures 0 .. S-2 and the B runs 1 .. S-1: the diagonal tiles hold 10
        #  jobs in 4 rows instead of 6 in 3)
        assert p2["pays"] and p2["tiles"] == 55 and p2["rows"] == 45 * 4 + 9 * 4 + 3
    twice = _capi.plan_job_tiles(jobs_of(np.concatenate([blocked, blocked])))
    assert twice["pays"] and twice["tiles"] == 110
    # a rank's contiguous share starts and ends inside tiles
    share = blocked[batch.contiguous_share(len(blocked), 1, 3)]
    assert _capi.plan_job_tiles(jobs_of(share))["pays"]
    # frame 0 against the other frames: tiles of a single row
    frames = _capi.plan_job_tiles(jobs_of([(0, f) for f in range(1, 65)]))
    assert not frames["pays"] and frames["tiles"] == 16 and frames["rows"] == 16
    # jobs of different sizes are never tiled
    uneven = jobs_of(blocked)
    uneven["n"][5] = n - 1
    assert not _capi.plan_job_tiles(uneven)["pays"]
    assert _capi.plan_job_tiles(jobs_of([]))["tiles"] == 0
    # nor are lists of fewer than 4 equal jobs
    for k in (1, 2, 3):
        few = _capi.plan_job_tiles(jobs_of(blocked[:k]))
        assert not few["pays"] and few["tiles"] == 0 and few["rows"] == 0
