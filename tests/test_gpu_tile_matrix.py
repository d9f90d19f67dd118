"""score_tile_kernel across what it can launch: both instantiations (8 count rows per warp for C <= 8, 16 for
C = 9..16, with its two-word histogram), replicated, partly replicated and unreplicated count tables, 6 / 7 / 8 teams,
claimed runs of other lengths than 8 units, chunks close to the 128 events of the 8-bit histogram fields, every
weight-function key with a tail term that carries weight, environments that hold only the anchor, and the
unknown-category check of the 16-row form.

Every GPU case lists an ensemble's jobs in batch.blocked_pairs order (or all pairs of two environment sets), asserts
that the list tiles, reads the launch geometry from the host query locohd_tile_geometry at the real largest
environments and asserts the intended (cp, rep_n, teams), asserts a tile launch, and compares every per-anchor score
with the CPU oracle (1e-9), with the one-pair-per-warp kernel on the same jobs (1e-12: same arithmetic, other chunk
boundaries) and the job means with numpy.  Launch switches that only move work or copy table entries must not change
a bit.  The CPU tests at the bottom pin the geometry rules themselves.
"""
import os

import numpy as np
import pytest

from benchdata import synth
from helpers import SCORE_TOL, assert_scores_close, set_both
from loco_hd_b200 import _capi, batch
from test_gpu_fuzz import WFS

JOB = [("a_first", "<u8"), ("b_first", "<u8"), ("n", "<u8")]
ACCEPT_OTHERS = {"accept_same": False}
B200_SMS = 148


# ---- fixtures and helpers -------------------------------------------------------------------------------------------
def _members(base, n_members, delta, seed):
    return [synth.partner(base, delta, seed + i) for i in range(n_members)]


def _ball(seed, n, C, radius, first_share=None):
    """n primitives uniform in a ball, one tag each; categories uniform over C, or category 0 for `first_share` of
    them and the others uniform over 1..C-1.  Every category occurs."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    xyz = d * (radius * rng.random(n) ** (1.0 / 3.0))[:, None]
    if first_share is None:
        cat = np.arange(n) % C
    else:
        cat = np.where(np.arange(n) < int(first_share * n), 0, 1 + np.arange(n) % max(C - 1, 1))
    cat = rng.permutation(cat).astype(np.uint16)
    return synth.Cloud(xyz, cat, np.arange(n, dtype=np.uint32), 1)


def _grid_pairs(n_a, n_b):
    """All (i, j) of two environment sets, in 4 x 4 blocks."""
    return np.array([(i, j) for bi in range(0, n_a, 4) for bj in range(0, n_b, 4)
                     for i in range(bi, min(bi + 4, n_a)) for j in range(bj, min(bj + 4, n_b))], dtype=np.int64)


def _env_offsets(env):
    """Environment offsets of an environment set (locohd_envset_dump without distances and categories)."""
    off = np.empty(len(env) + 1, np.uint64)
    env.ctx._check(env.ctx.lib.locohd_envset_dump(env.ctx.h, env.h, _capi._p(off), None, None, None))
    return off


class _Ensemble:
    """Structures and environments resident on the device; rows from clouds_a, columns from clouds_b (None: the same
    environment set on both sides, jobs in blocked_pairs order)."""

    def __init__(self, ctx, clouds_a, anchors_a, threshold, clouds_b=None, anchors_b=None):
        self.ctx, self.threshold = ctx, threshold
        self.clouds_a, self.anchors_a = clouds_a, np.asarray(anchors_a, np.uint32)
        self.st_a, self.env_a = self._build(clouds_a, self.anchors_a)
        if clouds_b is None:
            self.clouds_b, self.anchors_b, self.st_b, self.env_b = clouds_a, self.anchors_a, None, self.env_a
            self.pairs = batch.blocked_pairs(len(clouds_a), 4)
        else:
            self.clouds_b, self.anchors_b = clouds_b, np.asarray(anchors_b, np.uint32)
            self.st_b, self.env_b = self._build(clouds_b, self.anchors_b)
            self.pairs = _grid_pairs(len(clouds_a), len(clouds_b))
        self.n = len(self.anchors_a)
        assert len(self.anchors_b) == self.n
        self.jobs = np.array([(i * self.n, j * self.n, self.n) for i, j in self.pairs], dtype=JOB)
        self.sizes_a = self._sizes(self.env_a, len(clouds_a))
        self.sizes_b = self.sizes_a if clouds_b is None else self._sizes(self.env_b, len(clouds_b))
        self.max_a, self.max_b = int(self.sizes_a.max()), int(self.sizes_b.max())

    def _build(self, clouds, anchors):
        offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
        st = self.ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]),
                                     np.concatenate([c.cat for c in clouds]), np.concatenate([c.tag for c in clouds]))
        a_struct = np.repeat(np.arange(len(clouds), dtype=np.uint32), len(anchors))
        return st, self.ctx.envset_build(st, np.tile(anchors, len(clouds)), self.threshold, anchor_struct=a_struct)

    def _sizes(self, env, n_structs):
        return np.diff(_env_offsets(env)).astype(np.int64).reshape(n_structs, -1)   # [structure, anchor]

    def geometry(self, C):
        return _capi.tile_geometry(C, self.max_a, self.max_b)

    def score(self, expect_tiles=True):
        before = self.ctx.tile_launches
        res = self.ctx.score_jobs_stats(self.env_a, self.env_b, self.jobs, scores=True, job_means=True)
        used = self.ctx.tile_launches - before
        assert (used > 0) == expect_tiles, f"tile kernel launches: {used}"
        return res

    def oracle(self, oracle_mod, op):
        """[jobs, anchors] of the oracle; repeated anchors are scored once."""
        out = np.empty((len(self.pairs), self.n))
        an = np.stack([self.anchors_a, self.anchors_b], axis=1)
        uniq, inv = np.unique(an, axis=0, return_inverse=True)
        for k, (i, j) in enumerate(self.pairs.tolist()):
            a, b = self.clouds_a[i], self.clouds_b[j]
            out[k] = oracle_mod.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, uniq,
                                                self.threshold)[inv.ravel()]
        return out

    def close(self):
        for h in (self.env_b if self.st_b is not None else None, self.st_b, self.env_a, self.st_a):
            if h is not None:
                h.close()


def _check(ens, oracle_mod, op, monkeypatch, C, expect, label):
    """The list tiles, the geometry is `expect` (a dict of locohd_tile_geometry fields), the tile kernel scores it
    (teams >= 6) or does not (teams < 6); scores against the oracle, the pair kernel and numpy."""
    assert _capi.plan_job_tiles(ens.jobs)["pays"]
    g = ens.geometry(C)
    print(f"{label}: C={C} max_a={ens.max_a} max_b={ens.max_b} geometry={g} jobs={len(ens.jobs)} anchors={ens.n}")
    assert {k: g[k] for k in expect} == expect, g
    takes = g["teams"] >= 6
    tiled = ens.score(expect_tiles=takes)
    got = tiled["scores"].reshape(len(ens.pairs), ens.n)
    want = ens.oracle(oracle_mod, op)
    assert_scores_close(got.ravel(), want.ravel())
    monkeypatch.setenv("LOCOHD_NO_TILES", "1")
    plain = ens.score(expect_tiles=False)
    monkeypatch.delenv("LOCOHD_NO_TILES")
    assert np.abs(tiled["scores"] - plain["scores"]).max() <= 1e-12
    assert np.abs(tiled["job_means"] - want.mean(axis=1)).max() <= SCORE_TOL
    assert np.abs(tiled["job_means"] - got.mean(axis=1)).max() <= 1e-12
    return tiled, plain, want, g


# ---- a. category count across the instantiation boundary ------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 2, 8, 9, 12, 16], ids=lambda c: f"C{c}-cp{8 if c <= 8 else 16}")
def test_category_counts_across_the_instantiations(gpu_ctx, oracle_mod, monkeypatch, C):
    """Every category occurs (8..15 too for C = 16).  C = 2: 95 % of one category, single counts in the hundreds.
    C = 1: identical compositions everywhere, every score 0 up to the rounding of the difference form."""
    rng = np.random.default_rng(100 + C)
    base = synth.gen(40 + C, 150, 3, C)
    threshold = 10.0
    if C == 2:
        base.cat[:] = (rng.random(base.n) < 0.05).astype(np.uint16)
        threshold = 13.0
    members = _members(base, 9, 1.0, 1000 + 10 * C)
    assert np.array_equal(np.unique(base.cat), np.arange(C))
    anchors = np.arange(0, base.n, 5, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, C, [("uniform", (3.0, 10.0))], tag_rule=ACCEPT_OTHERS)
    ens = _Ensemble(gpu_ctx, members, anchors, threshold)
    assert ens.max_a < 300
    expect = {"cp": 8, "rep_n": 64, "teams": 8} if C <= 8 else {"cp": 16, "rep_n": 0, "teams": 8}
    tiled, _, want, _ = _check(ens, oracle_mod, op, monkeypatch, C, expect, f"a C={C}")
    if C == 1:
        # The oracle normalises both sides to the composition (1.0) and scores exactly 0.  The kernels give exact 0 only
        # where the counts are equal (no mismatch); otherwise H comes from the difference form sqrt(a) / sqrt(nA) -
        # sqrt(b) / sqrt(nB) with both products rounded, a residue of ~1e-16 per step (measured on a B200: ~1e-17).
        assert np.all(want == 0.0)
        assert np.abs(tiled["scores"]).max() <= 1e-15
    else:
        assert want.max() > 0.0
    if C == 2:
        assert ens.max_a > 150   # the majority category alone counts well over 100 in the largest environments
    ens.close()


# ---- b. the same data through both instantiations --------------------------------------------------------------------
@pytest.mark.gpu
def test_extra_category_rows_add_exact_zeros(gpu_ctx, oracle_mod, monkeypatch):
    """Structures whose categories are 0..7, scored as C = 8 (8 rows) and C = 12 (16 rows): the four empty rows add
    fma(0, 0, D) = D and 0 to the difference form and never count as a mismatch, so the scores are bit-identical.
    Categories mapped 0..7 -> 15..8 with C = 16: the rows are summed in another order, nothing else changes."""
    base = synth.gen(51, 110, 4, 8)
    members = _members(base, 9, 1.2, 5100)
    anchors = np.arange(1, base.n, 4, dtype=np.uint32)
    res = {}
    for C in (8, 12):
        op = set_both(gpu_ctx, oracle_mod, C, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule=ACCEPT_OTHERS)
        ens = _Ensemble(gpu_ctx, members, anchors, 10.0)
        expect = {"cp": 8, "rep_n": 64, "teams": 8} if C == 8 else {"cp": 16, "rep_n": 0, "teams": 8}
        res[C] = _check(ens, oracle_mod, op, monkeypatch, C, expect, f"b C={C}")[0]
        ens.close()
    assert np.array_equal(res[8]["scores"], res[12]["scores"])
    flipped = [synth.Cloud(m.xyz, (15 - m.cat).astype(np.uint16), m.tag, m.k) for m in members]
    op = set_both(gpu_ctx, oracle_mod, 16, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule=ACCEPT_OTHERS)
    ens = _Ensemble(gpu_ctx, flipped, anchors, 10.0)
    res16 = _check(ens, oracle_mod, op, monkeypatch, 16, {"cp": 16, "rep_n": 0, "teams": 8}, "b C=16 flipped")[0]
    assert np.abs(res16["scores"] - res[8]["scores"]).max() <= 1e-12
    ens.close()


# ---- c. replicated, partly replicated and unreplicated tables --------------------------------------------------------
@pytest.mark.gpu
def test_replicated_tables_copy_entries_only(gpu_ctx, oracle_mod, monkeypatch):
    """Category counts far above 64: look-ups of entries below and at or above rep_n (the mixed addressing) and of the
    unreplicated tables.  LOCOHD_TILE_REP unset (64), 0 (score_tile_kernel<8, false>), 1 and 16: bit-identical."""
    rng = np.random.default_rng(61)
    base = synth.gen(61, 150, 3, 3)
    base.cat[:] = np.where(rng.random(base.n) < 0.9, 0, rng.integers(1, 3, base.n)).astype(np.uint16)
    members = _members(base, 9, 1.0, 6100)
    anchors = np.arange(0, base.n, 4, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 3, [("uniform", (3.0, 12.0))], tag_rule=ACCEPT_OTHERS)
    ens = _Ensemble(gpu_ctx, members, anchors, 12.0)
    assert ens.max_a >= 140   # category 0 holds 90 % of the members: counts up to twice rep_n
    ref = _check(ens, oracle_mod, op, monkeypatch, 3, {"cp": 8, "rep_n": 64, "teams": 8}, "c REP unset")[0]
    for rep in (0, 1, 16):
        monkeypatch.setenv("LOCOHD_TILE_REP", str(rep))
        g = ens.geometry(3)
        print(f"c REP={rep}: geometry={g}")
        assert (g["cp"], g["rep_n"], g["teams"]) == (8, rep, 8)
        got = ens.score()
        assert np.array_equal(got["scores"], ref["scores"]), f"LOCOHD_TILE_REP={rep}"
        assert np.array_equal(got["job_means"], ref["job_means"])
    monkeypatch.delenv("LOCOHD_TILE_REP")
    ens.close()


# ---- d. teams and claimed runs ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_team_counts_and_run_lengths(gpu_ctx, oracle_mod, monkeypatch):
    """20 structures of 203 primitives, every primitive 21 times an anchor: 15 tiles x 4263 anchors = 63 945 units, so
    that even a run of 13 units is what the launch claims (run = min(LOCOHD_TILE_RUN, units / (4 x CTAs x teams)),
    148 CTAs on a B200).  6 and 7 teams, runs of 1, 3 and 13 units in tile-major order and in slices of 100 anchors
    (runs that cross tiles, slices and the end of the unit list): bit-identical to the default launch.  5 teams: the
    tile kernel is not taken."""
    base = synth.gen(31, 29, 7, 7)
    assert base.n == 203
    members = _members(base, 20, 1.5, 3100)
    anchors = np.tile(np.arange(base.n, dtype=np.uint32), 21)
    op = set_both(gpu_ctx, oracle_mod, 7, [("hyper_exp", (1.0, 0.2))], tag_rule=ACCEPT_OTHERS)
    ens = _Ensemble(gpu_ctx, members, anchors, 10.0)
    plan = _capi.plan_job_tiles(ens.jobs)
    units = plan["tiles"] * ens.n
    assert plan["tiles"] == 15 and units // (B200_SMS * 8 * 4) >= 13
    ref, plain, _, _ = _check(ens, oracle_mod, op, monkeypatch, 7, {"cp": 8, "rep_n": 64, "teams": 8}, "d default")
    for teams in (7, 6):
        monkeypatch.setenv("LOCOHD_TILE_TEAMS", str(teams))
        g = ens.geometry(7)
        print(f"d TEAMS={teams}: geometry={g}")
        assert (g["cp"], g["teams"]) == (8, teams) and g["rep_n"] == 64
        assert np.array_equal(ens.score()["scores"], ref["scores"]), f"LOCOHD_TILE_TEAMS={teams}"
    monkeypatch.setenv("LOCOHD_TILE_TEAMS", "5")
    assert ens.geometry(7)["teams"] == 5
    assert np.array_equal(ens.score(expect_tiles=False)["scores"], plain["scores"])
    monkeypatch.delenv("LOCOHD_TILE_TEAMS")
    for run in (1, 3, 13):
        for sl in ("0", "100"):
            monkeypatch.setenv("LOCOHD_TILE_RUN", str(run))
            monkeypatch.setenv("LOCOHD_TILE_SLICE", sl)
            got = ens.score()
            print(f"d RUN={run} SLICE={sl}: bit-identical={np.array_equal(got['scores'], ref['scores'])}")
            assert np.array_equal(got["scores"], ref["scores"]), f"LOCOHD_TILE_RUN={run} LOCOHD_TILE_SLICE={sl}"
            assert np.array_equal(got["job_means"], ref["job_means"])
    monkeypatch.delenv("LOCOHD_TILE_RUN")
    monkeypatch.delenv("LOCOHD_TILE_SLICE")
    ens.close()


# ---- e. the largest environments the tile kernel takes ---------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C,n,expect", [
    (8, 500, {"cp": 8, "rep_n": 0, "teams": 6}),      # score_tile_kernel<8, false>: no room left for replication
    (12, 445, {"cp": 16, "rep_n": 0, "teams": 6}),
    (8, 506, {"cp": 8, "teams": 5}),                  # just past the bound: the pair kernel scores it
], ids=["C8-500-teams6-rep0", "C12-445-teams6", "C8-506-teams5-no-tiles"])
def test_largest_environments(gpu_ctx, oracle_mod, monkeypatch, C, n, expect):
    """Every primitive within the threshold of every other: each environment holds the whole structure, chunks of
    (max_a + max_b - 2) / 8 >= 110 events, close to the 128 the 8-bit histogram fields hold.  C = 8 with 40 % of one
    category: counts of 200 in the unreplicated tables."""
    base = _ball(70 + C, n, C, 4.0, first_share=0.4 if C == 8 else None)
    assert np.array_equal(np.unique(base.cat), np.arange(C))
    members = _members(base, 8, 0.3, 7000 + n)
    anchors = np.arange(3, n, n // 24, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, C, [("uniform", (3.0, 10.0))], tag_rule=ACCEPT_OTHERS)
    ens = _Ensemble(gpu_ctx, members, anchors, 14.0)
    assert ens.max_a == ens.max_b == n and np.all(ens.sizes_a == n)
    assert (ens.max_a + ens.max_b - 2) / 8 >= 110
    _check(ens, oracle_mod, op, monkeypatch, C, expect, f"e C={C} n={n}")
    ens.close()


# ---- f. weight functions ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_weight_function_keys(gpu_ctx, oracle_mod, monkeypatch):
    """The W-keyed store of every weight function of the fuzz test (uniform, kumaraswamy with integer and generic
    exponents, hyper_exp, dagum), threshold 8 A, where most of them have W(threshold) well below 1: the tail
    w_inf - W(last) of the last chunk carries weight.  C alternates between the two instantiations."""
    threshold = 8.0
    tails = [oracle_mod.wf_integral_point(name, q, threshold) for name, q in WFS]
    assert min(tails) < 0.5 and sum(t < 0.9 for t in tails) >= 4
    for k, (name, q) in enumerate(WFS):
        C = 6 if k % 2 == 0 else 11
        base = synth.gen(80 + k, 80, 5, C)
        members = _members(base, 8, 1.2, 8000 + 10 * k)
        anchors = np.arange(k % 3, base.n, 3, dtype=np.uint32)
        op = set_both(gpu_ctx, oracle_mod, C, [(name, q)], tag_rule=ACCEPT_OTHERS)
        ens = _Ensemble(gpu_ctx, members, anchors, threshold)
        expect = {"cp": 8 if C <= 8 else 16, "teams": 8}
        _check(ens, oracle_mod, op, monkeypatch, C, expect, f"f {name}{tuple(q)} W(thr)={tails[k]:.3f}")
        ens.close()


# ---- g. sparse members -----------------------------------------------------------------------------------------------
def _sparse_base(seed, C):
    """Sites 15 A apart, 6 A threshold: a site holds 1 (70 %), 2 (25 %) or 3 primitives within 1.2 A."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.arange(6) * 15.0] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    per_site = rng.choice([1, 2, 3], size=len(g), p=[0.7, 0.25, 0.05])
    xyz = np.repeat(g, per_site, axis=0) + rng.uniform(-0.7, 0.7, size=(per_site.sum(), 3))
    n = len(xyz)
    return synth.Cloud(xyz, rng.integers(0, C, n).astype(np.uint16), np.arange(n, dtype=np.uint32), 1)


@pytest.mark.gpu
def test_sparse_members(gpu_ctx, oracle_mod, monkeypatch):
    """Most anchors see only themselves or one neighbour: units whose 8 staged environments all hold the anchor only
    (no bulk copy at all, the member stored by hand), and odd and even sizes side by side."""
    C = 5
    base = _sparse_base(91, C)
    members = _members(base, 8, 0.1, 9100)
    anchors = np.arange(base.n, dtype=np.uint32)
    op = set_both(gpu_ctx, oracle_mod, C, [("uniform", (0.0, 6.0))], tag_rule=ACCEPT_OTHERS)
    ens = _Ensemble(gpu_ctx, members, anchors, 6.0)
    s = ens.sizes_a
    assert set(np.unique(s).tolist()) == {1, 2, 3} and np.mean(s <= 2) > 0.8
    assert np.all(s == s[0]) and np.count_nonzero(s[0] == 1) > 100   # anchor p has the same size in all 8 structures
    assert [tuple(p) for p in ens.pairs[:22].tolist()] == [(i, j) for i in range(4) for j in range(4) if i < j] + \
        [(i, j) for i in range(4) for j in range(4, 8)]   # the second tile: rows 0..3 against columns 4..7
    tiled, _, want, _ = _check(ens, oracle_mod, op, monkeypatch, C, {"cp": 8, "rep_n": 64, "teams": 8}, "g sparse")
    assert want.max() > 0.0 and np.all(tiled["scores"].reshape(len(ens.pairs), -1)[:, s[0] == 1] == 0.0)
    ens.close()


# ---- h. unknown categories in the 16-row form ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("where", ["member", "anchor"])
def test_unknown_category_with_sixteen_rows(gpu_ctx, oracle_mod, monkeypatch, where):
    """C = 12 (score_tile_kernel<16, false>): a category the instance does not know inside an environment (13: a
    field of the second histogram word that has to stay empty), or as the anchor of an environment that holds only the
    anchor (an isolated primitive far from the structure).  Both: status 3 from a tile launch.  Without them the
    same ensemble scores cleanly."""
    C = 12
    base = synth.gen(24, 40, 8, C)
    far = synth.Cloud(np.array([[500.0, 500.0, 500.0]]), np.zeros(1, np.uint16), np.array([10 ** 6], np.uint32), 1)
    base = synth.Cloud(np.vstack([base.xyz, far.xyz]), np.r_[base.cat, far.cat].astype(np.uint16),
                       np.r_[base.tag, far.tag].astype(np.uint32), base.k)
    members = _members(base, 8, 1.0, 2400)
    anchors = np.r_[np.arange(0, base.n - 1, 2), base.n - 1].astype(np.uint32)
    op = set_both(gpu_ctx, oracle_mod, C, [("uniform", (3.0, 10.0))], tag_rule=ACCEPT_OTHERS)
    ens = _Ensemble(gpu_ctx, members, anchors, 10.0)
    assert np.all(ens.sizes_a[:, -1] == 1)
    _check(ens, oracle_mod, op, monkeypatch, C, {"cp": 16, "rep_n": 0, "teams": 8}, f"h clean ({where})")
    ens.close()
    if where == "member":
        members[5].cat[17] = 13
    else:
        members[3].cat[base.n - 1] = _capi.UNKNOWN_CATEGORY
    ens = _Ensemble(gpu_ctx, members, anchors, 10.0)
    assert ens.geometry(C)["cp"] == 16 and _capi.plan_job_tiles(ens.jobs)["pays"]
    before = gpu_ctx.tile_launches
    with pytest.raises(_capi.LocoHDError) as ei:
        gpu_ctx.score_jobs_stats(ens.env_a, ens.env_b, ens.jobs, scores=True)
    assert ei.value.status == 3 and gpu_ctx.tile_launches > before
    ens.close()


# ---- i. randomised tile cases ----------------------------------------------------------------------------------------
def _fuzz_case(rng, case):
    C = int(rng.integers(1, 17))
    wf = WFS[int(rng.integers(len(WFS)))]
    threshold = float(rng.uniform(6.0, 15.0))

    def ensemble(seed, n_members):
        base = synth.gen(seed, int(rng.integers(20, 90)), int(rng.integers(2, 9)), C)
        return base, _members(base, n_members, float(rng.uniform(0.3, 2.0)), seed * 100)

    base_a, members_a = ensemble(5000 + 2 * case, int(rng.integers(8, 13)))
    two_sets = bool(rng.random() < 0.4)
    if two_sets:
        base_b, members_b = ensemble(5001 + 2 * case, int(rng.integers(4, 9)))
        n = int(rng.integers(4, min(base_a.n, base_b.n, 60) + 1))
        anchors_b = np.sort(rng.choice(base_b.n, n, replace=False))
    else:
        members_b = None
        n = int(rng.integers(4, min(base_a.n, 80) + 1))
        anchors_b = None
    anchors_a = np.sort(rng.choice(base_a.n, n, replace=False))
    return C, wf, threshold, members_a, anchors_a, members_b, anchors_b


@pytest.mark.gpu
def test_random_tile_cases(gpu_ctx, oracle_mod, monkeypatch):
    """Seeded: member count, C in [1, 16], weight function, threshold 6..15 A, anchor subset, one environment set or
    two.  Cases the tile kernel does not take (the list does not tile, or fewer than 6 teams fit) are skipped and
    counted.  LOCOHD_TILE_FUZZ_CASES raises the number of cases (default 12)."""
    rng = np.random.default_rng(20261020)
    n_cases = int(os.environ.get("LOCOHD_TILE_FUZZ_CASES", "12"))
    executed, skipped, cps = 0, 0, set()
    for case in range(n_cases):
        C, wf, threshold, members_a, anchors_a, members_b, anchors_b = _fuzz_case(rng, case)
        op = set_both(gpu_ctx, oracle_mod, C, [wf], tag_rule=ACCEPT_OTHERS)
        ens = _Ensemble(gpu_ctx, members_a, anchors_a, threshold, members_b, anchors_b)
        g = ens.geometry(C)
        if not _capi.plan_job_tiles(ens.jobs)["pays"] or g["teams"] < 6:
            skipped += 1
            ens.close()
            continue
        expect = {"cp": 8 if C <= 8 else 16, "teams": g["teams"]}
        _check(ens, oracle_mod, op, monkeypatch, C, expect, f"i case {case} {wf[0]} thr={threshold:.2f} "
                                                            f"sets={1 if members_b is None else 2}")
        cps.add(g["cp"])
        executed += 1
        ens.close()
    print(f"random tile cases: {executed} scored, {skipped} skipped (not tile-eligible), cp {sorted(cps)}")
    assert executed >= n_cases // 2 and cps == {8, 16}


# ---- CPU: the geometry rules -----------------------------------------------------------------------------------------
def test_geometry_instantiation_by_category_count():
    """C <= 8: 8 count rows per warp with replicated tables at small environments; C = 9..16: 16 rows, never
    replicated; C = 17 (and 0): no tile kernel."""
    for C in range(1, 9):
        assert _capi.tile_geometry(C, 100, 120) == {"teams": 8, "cp": 8, "rep_n": 64, "table_n": 128}
    for C in range(9, 17):
        for m in (1, 100, 300, 445):
            g = _capi.tile_geometry(C, m, m)
            assert g["cp"] == 16 and g["rep_n"] == 0 and g["teams"] >= 6
    for C in (0, 17, 255):
        assert _capi.tile_geometry(C, 100, 100)["teams"] == 0


def test_geometry_environment_size_limits():
    """max_a + max_b > 1024 (more than 128 events in a lane's chunk) or an empty side: no tile kernel."""
    for C in (4, 12):
        assert _capi.tile_geometry(C, 512, 512)["teams"] > 0
        assert _capi.tile_geometry(C, 512, 513)["teams"] == 0
        assert _capi.tile_geometry(C, 1000, 25)["teams"] == 0
        assert _capi.tile_geometry(C, 0, 10)["teams"] == 0
        assert _capi.tile_geometry(C, 10, 0)["teams"] == 0
    assert _capi.tile_geometry(3, 1, 1) == {"teams": 8, "cp": 8, "rep_n": 64, "table_n": 64}


def test_geometry_six_team_bound():
    """Where the launch changes shape as both sides grow: C <= 8 keeps 6 teams up to 505 members (without table
    replication from 496 on), C = 9..16 up to 445; one member more leaves 5 teams, and the jobs take the pair kernel."""
    g8 = {m: _capi.tile_geometry(8, m, m) for m in (361, 362, 369, 370, 427, 428, 495, 496, 505, 506)}
    assert (g8[361]["teams"], g8[361]["rep_n"]) == (8, 17)
    assert (g8[362]["teams"], g8[362]["rep_n"]) == (8, 0)
    assert (g8[369]["teams"], g8[370]["teams"]) == (8, 7)
    assert (g8[427]["teams"], g8[428]["teams"]) == (7, 6)
    assert (g8[495]["teams"], g8[495]["rep_n"]) == (6, 18)
    assert (g8[496]["teams"], g8[496]["rep_n"]) == (6, 0)
    assert (g8[505]["teams"], g8[505]["rep_n"]) == (6, 0)
    assert g8[506]["teams"] == 5
    g12 = {m: _capi.tile_geometry(12, m, m)["teams"] for m in (307, 308, 367, 368, 445, 446)}
    assert g12 == {307: 8, 308: 7, 367: 7, 368: 6, 445: 6, 446: 5}
    # the case (e) shapes of the GPU tests: >= 110 events per lane's chunk at 6 teams
    assert (500 + 500 - 2) / 8 >= 110 and (445 + 445 - 2) / 8 >= 110


def test_geometry_overrides_only_lower(monkeypatch):
    """LOCOHD_TILE_TEAMS lowers the team count and LOCOHD_TILE_REP the replicated entries; team counts at or above the
    default, zero, negative or garbage and table counts at or above the default or negative change nothing.  Fewer teams leave more shared memory over, which may
    replicate more of the tables."""
    shapes = [(8, 100, 100), (8, 365, 365), (8, 500, 500), (12, 200, 200), (12, 440, 440), (3, 1, 1)]
    default = {s: _capi.tile_geometry(*s) for s in shapes}
    for t in ("-3", "0", "1", "4", "5", "6", "7", "8", "9", "64", "x"):
        monkeypatch.setenv("LOCOHD_TILE_TEAMS", t)
        for s in shapes:
            g, d = _capi.tile_geometry(*s), default[s]
            want = int(t) if t.lstrip("-").isdigit() and 1 <= int(t) < d["teams"] else d["teams"]
            assert g["teams"] == want, (t, s)
            assert (g["cp"], g["table_n"]) == (d["cp"], d["table_n"])
            assert g["rep_n"] >= d["rep_n"] and (d["cp"] == 8 or g["rep_n"] == 0)
    monkeypatch.delenv("LOCOHD_TILE_TEAMS")
    for r in ("-1", "0", "1", "16", "63", "64", "65", "1000"):
        monkeypatch.setenv("LOCOHD_TILE_REP", r)
        for s in shapes:
            g, d = _capi.tile_geometry(*s), default[s]
            want = int(r) if r.lstrip("-").isdigit() and 0 <= int(r) < d["rep_n"] else d["rep_n"]
            assert g["rep_n"] == want, (r, s)
            assert {k: g[k] for k in ("teams", "cp", "table_n")} == {k: d[k] for k in ("teams", "cp", "table_n")}
    monkeypatch.setenv("LOCOHD_TILE_TEAMS", "5")
    assert _capi.tile_geometry(8, 500, 500)["rep_n"] == 64   # one team less: 40 KB more for the tables
