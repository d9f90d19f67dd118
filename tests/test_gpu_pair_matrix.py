"""The pair route (one warp per anchor pair: score_fast_kernel, score_kernel for everything the fast kernel does not
take) across what it can launch: the 8 instantiations of score_fast_kernel<CP, KEY_IS_W, WEIGHTED>, score_kernel at
category counts up to 255 staged with several warps, staged with one warp and unstaged, the split of one call between
the fast kernel and a second score_kernel pass at the stage boundary, the backward walk score_grad_kernel at large C,
the from_anchors walk at 255 categories and the category-count limits of the API.

Every case of the two scoring kernels scores resident environment sets with explicit pairs (locohd_score_pairs, host
pair lists and weight function indices: the launch count moves only by what launch_score starts), restates the launch
rules below to say which route and geometry it means to hit, prints it, asserts the launch count of that route and that
no tile kernel ran, and compares every score with the CPU oracle (1e-9).  The gradient cases compare with the CPU
references of the gradient tests and count the launches of the plain call on the same input.  Where two routes do
the same arithmetic on the same keys the scores must be bit-identical.  The CPU tests at the bottom pin the restated
rules.
"""
import numpy as np
import pytest

import grad_reference as gr
import rows_grad_reference as rr
from benchdata import synth
from helpers import assert_scores_close, set_both
from loco_hd_b200 import _capi
from test_gpu_tile_matrix import _ball

GRAD_TOL = 1e-9     # the bars of test_gpu_grad.py / test_gpu_rows_grad.py
ROUTE_TOL = 1e-12
HELL2 = ("Hellinger", (2.0,))
SDS = [   # test_gpu_parity.SDS
    ("Hellinger", (2.0,)),
    ("Hellinger", (3.4277149325231795,)),
    ("Kolmogorov-Smirnov", ()),
    ("Kullback-Leibler", (3.241633447825855,)),
    ("Renyi", (2.3, 0.7)),
    ("Renyi", (1.0, 0.5)),
    ("Renyi", (0.0, 0.5)),
    ("Renyi", (float("inf"), 0.5)),
]
# W(threshold) < 1 for the first two at thresholds of 10-12 A: the tail term w_inf - W(last) carries weight
WFS3 = [("kumaraswamy", (3.0, 14.0, 2.0, 5.0)), ("hyper_exp", (1.0, 0.1)), ("uniform", (2.0, 9.0))]
WF1 = [WFS3[0]]
ACCEPT_OTHERS = {"accept_same": False}   # every other primitive within the threshold is a member


# ---- the launch rules of the pair route, restated from loco_hd_b200/csrc/locohd_kernels.cu -------------------------
SCORE_BUDGET = 100 * 1024   # launch_generic: shared memory of a score_kernel CTA (:3053)
SCORE_MAX_WARPS = 8         # kScoreMaxWarps (:1316)
STAGE_MAX = 2048            # the largest stage of either kernel (:3055, :3209)


def _pad(m):
    return (int(m) + 1) & ~1


def _round64(x):
    return (int(x) + 63) & ~63


def score_state_bytes(C):   # :1323, per-lane values and counts of score_kernel + its mbarrier
    return (((2 * C * 32 * 8 + 2 * C * 32 * 4) + 15) & ~15) + 16


def grad_state_bytes(C):    # :1584
    return ((2 * C * 32 * 8 + 2 * C * 32 * 4) + 15) & ~15


def fast_max_warps(key_is_w, weighted):   # score_fast_max_warps (:1319)
    return 24 if weighted else (32 if key_is_w else 28)


def generic_launch(C, hell2, stage_want):
    """launch_generic (:3050-3067): the stage (0: every pair read from global memory), warps per CTA, shared memory."""
    state = score_state_bytes(C)
    cap = min(stage_want, STAGE_MAX)
    per_warp = state + 8 * cap
    if per_warp > SCORE_BUDGET:
        cap, per_warp = 0, state
    assert per_warp <= 220 * 1024
    warps = max(1, min(SCORE_MAX_WARPS, SCORE_BUDGET // per_warp))
    return {"kernel": f"score_kernel<{str(hell2).lower()}>", "stage_cap": cap, "warps": warps, "smem": per_warp * warps}


def fast_stage(pad_max, mean_a, mean_b):
    """launch_score (:3205-3211): everything when the largest pair is small, else what a typical pair needs."""
    if pad_max <= 1024:
        return pad_max
    return min(_round64(int(1.5 * (mean_a + mean_b)) + 64), STAGE_MAX, pad_max)


def pair_route(C, hell2, unit_w, key_is_w, max_a, max_b, mean_a, mean_b):
    """launch_score (:3192-3237) for explicit pairs.  max_* and mean_* are the environment sets' largest and mean
    environment sizes.  The launch takes its mean from the entries the store holds, which is at least the member count
    (the fused gather reserves its store in chunks of 2048 entries), so a stage that depends on the mean is not known
    from the sizes; the cases here either keep pad_max <= 1024 or reach the 2048 cap with the members alone."""
    pad_max = _pad(max_a) + _pad(max_b)
    if not (hell2 and C <= 16):
        return {"launches": 1, "pad_max": pad_max, "generic": generic_launch(C, hell2, pad_max)}
    stage = fast_stage(pad_max, mean_a, mean_b)
    assert stage == fast_stage(pad_max, 1e9, 1e9), "the stage would depend on the store's fill"
    table_n = _round64(min(max(max_a, max_b) + 2, stage))
    cp = 8 if C <= 8 else 16
    per_warp = cp * 32 * 4 + 16 + (stage + 4) * 8
    warps = max(1, min(fast_max_warps(key_is_w, not unit_w), (220 * 1024 - 3 * table_n * 8 - 128) // per_warp))
    r = {"launches": 1 + (pad_max > stage), "pad_max": pad_max,
         "fast": f"score_fast_kernel<{cp}, {str(key_is_w).lower()}, {str(not unit_w).lower()}>",
         "stage": stage, "table_n": table_n, "warps": warps}
    if pad_max > stage:
        r["second"] = generic_launch(C, True, 0)   # only_unstaged = stage: the pairs above it, from global memory
    return r


# ---- fixtures and helpers -------------------------------------------------------------------------------------------
@pytest.fixture
def fresh_ctx():
    ctx = _capi.Context(0)
    yield ctx
    ctx.close()


def _params(ctx, oracle_mod, C, wfs, weights=None, sd=HELL2):
    return set_both(ctx, oracle_mod, C, wfs, weights, sd, tag_rule=ACCEPT_OTHERS)


def _cat_weights(C):
    """Uneven, positive, none of them 1."""
    w = 0.3 + (np.arange(C) * 0.618034) % 2.4
    assert np.all(w > 0) and np.all(w != 1.0) and (C == 1 or w.max() > 2 * w.min())
    return w


def _sparse_cloud(seed, n, side, C):
    rng = np.random.default_rng(seed)
    return synth.Cloud(rng.uniform(0.0, side, (n, 3)), rng.integers(0, C, n).astype(np.uint16),
                       np.arange(n, dtype=np.uint32), 1)


def _by_radius(cloud, step, offset=0):
    """Every step-th primitive in the order of its distance from the cloud's centre: environments of every size."""
    order = np.argsort(np.linalg.norm(cloud.xyz - cloud.xyz.mean(axis=0), axis=1), kind="stable")
    return order[offset::step].astype(np.uint32)


class _Set:
    """Environments of the anchors (structure, primitive) of several clouds, built on the device from one structure
    set after the parameters are set (categories are converted and the store is keyed when they are built)."""

    def __init__(self, ctx, clouds, anchors, threshold):
        self.ctx, self.clouds, self.threshold = ctx, clouds, threshold
        self.anchors = np.asarray(anchors, np.uint32).reshape(-1, 2)
        offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
        self.st = ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]),
                                     np.concatenate([c.cat for c in clouds]), np.concatenate([c.tag for c in clouds]))
        self.env = ctx.envset_build(self.st, self.anchors[:, 1], threshold, anchor_struct=self.anchors[:, 0])
        off = np.empty(len(self.anchors) + 1, np.uint64)
        ctx._check(ctx.lib.locohd_envset_dump(ctx.h, self.env.h, _capi._p(off), None, None, None))
        self.sizes = np.diff(off).astype(np.int64)
        self.max, self.mean = int(self.sizes.max()), float(self.sizes.mean())

    def close(self):
        self.env.close()
        self.st.close()


def _anchors(struct, prims):
    return np.stack([np.full(len(prims), struct, np.uint32), np.asarray(prims, np.uint32)], axis=1)


def _route(C, sd, weights, wfs, a, b):
    unit = weights is None or np.all(np.asarray(weights) == 1.0)
    return pair_route(C, tuple(sd) == HELL2, unit, len(wfs) == 1, a.max, b.max, a.mean, b.mean)


def _score(ctx, a, b, pairs, route, wf_idx=None, label=""):
    """score_pairs with the launch count of `route` and no tile launch."""
    print(f"{label}: pairs={len(pairs)} max_a={a.max} max_b={b.max} route={route}")
    before, tiles = ctx.launch_count, ctx.tile_launches
    got = ctx.score_pairs(a.env, b.env, np.asarray(pairs, np.uint32), wf_idx=wf_idx)
    assert ctx.launch_count - before == route["launches"], f"launches {ctx.launch_count - before}"
    assert ctx.tile_launches == tiles
    return got


def _oracle(oracle_mod, op, a, b, pairs, wf_idx=None, debug=False):
    """Oracle scores of environment pairs (index into a, index into b); with debug also the final category counts."""
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    sa, sb = a.anchors[pairs[:, 0]], b.anchors[pairs[:, 1]]
    out = np.empty(len(pairs))
    counts = np.zeros((len(pairs), 2, op.n_categories), np.int64)
    for s, t in {(int(x), int(y)) for x, y in zip(sa[:, 0], sb[:, 0])}:
        m = (sa[:, 0] == s) & (sb[:, 0] == t)
        A, B = a.clouds[s], b.clouds[t]
        r = oracle_mod.from_primitives(op, A.xyz, A.cat, A.tag, B.xyz, B.cat, B.tag,
                                       np.stack([sa[m, 1], sb[m, 1]], axis=1), a.threshold,
                                       wf_idx=None if wf_idx is None else np.asarray(wf_idx)[m], debug=True)
        out[m], counts[m] = r["scores"], r["counts"]
    return (out, counts) if debug else out


def _case(ctx, oracle_mod, C, sd, weights, wfs, sets, pairs, wf_idx=None, label="", expect=None):
    """Sets the parameters, builds the sets ([(clouds, anchors)], one or two), scores the pairs on the route the rules
    give (`expect`: fields of it the case is about) and against the oracle.  Returns (scores, oracle, route, sets,
    the oracle's final category counts [pair, side, category])."""
    op = _params(ctx, oracle_mod, C, wfs, weights, sd)
    built = [_Set(ctx, clouds, anchors, sets[0][2]) for clouds, anchors, _ in sets]
    a, b = built[0], built[-1]
    route = _route(C, sd, weights, wfs, a, b)
    if expect:
        flat = {**route, **route.get("generic", {})}
        assert {k: flat[k] for k in expect} == expect, route
    got = _score(ctx, a, b, pairs, route, wf_idx, f"{label} C={C} {sd[0]}{list(sd[1])} "
                                                   f"{'weighted' if weights is not None else 'unit'} wfs={len(wfs)}")
    want, counts = _oracle(oracle_mod, op, a, b, pairs, wf_idx, debug=True)
    assert_scores_close(got, want)
    return got, want, route, built, counts


def _close(built):
    for s in {id(x): x for x in built}.values():
        s.close()


# ---- a. the fast kernel's instantiations -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True], ids=["unit", "weighted"])
@pytest.mark.parametrize("key_is_w", [True, False], ids=["W-keyed", "distance-keyed"])
@pytest.mark.parametrize("C", [1, 8, 9, 16])
def test_fast_kernel_instantiations(gpu_ctx, oracle_mod, C, key_is_w, weighted):
    """score_fast_kernel<8 | 16, KEY_IS_W, WEIGHTED> at the smallest and largest C of either row count.  Every category
    occurs in the environments; distance-keyed: three weight functions chosen per pair."""
    base = synth.gen(200 + C, 90, 4, C)
    partner = synth.partner(base, 1.0, 2000 + C)
    anchors = np.arange(0, base.n, 2, dtype=np.uint32)
    n = len(anchors)
    wfs = WF1 if key_is_w else WFS3
    weights = _cat_weights(C) if weighted else None
    wf_idx = None if key_is_w else (np.arange(n) % 3).astype(np.uint32)
    pairs = np.stack([np.arange(n), n + np.arange(n)], axis=1)
    sets = [([base, partner], np.r_[_anchors(0, anchors), _anchors(1, anchors)], 10.0)]
    cp = 8 if C <= 8 else 16
    expect = {"launches": 1, "fast": f"score_fast_kernel<{cp}, {str(key_is_w).lower()}, {str(weighted).lower()}>"}
    got, want, _, built, counts = _case(gpu_ctx, oracle_mod, C, HELL2, weights, wfs, sets, pairs, wf_idx, "a", expect)
    assert np.all(counts.sum(axis=(0, 1)) > 0), "a category does not occur"
    assert C == 1 or want.max() > 0.05
    _close(built)


# ---- b. the same arithmetic across kernels and category counts -------------------------------------------------------
def _small_set16():
    base = synth.gen(300, 120, 4, 16)
    partner = synth.partner(base, 1.0, 3000)
    anchors = np.arange(0, base.n, 3, dtype=np.uint32)
    n = len(anchors)
    return [base, partner], np.r_[_anchors(0, anchors), _anchors(1, anchors)], n


def _large_set(C, seed):
    """A dense ball (2 400 primitives, radius 10 A, threshold 10 A) and a moved copy: environments of 700 - 2 300
    members, pairs of 1 400 - 4 600 keys.  Anchors every 40th primitive by distance from the centre."""
    base = _ball(seed, 2400, C, 10.0)
    partner = synth.partner(base, 0.5, seed + 1)
    anchors = _by_radius(base, 40, 7)
    return [base, partner], np.r_[_anchors(0, anchors), _anchors(1, anchors)], len(anchors)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["small", "large"])
def test_same_arithmetic_across_category_counts(gpu_ctx, oracle_mod, which):
    """Structures with categories 0..15.  C = 16 (score_fast_kernel<16, ...>) and C = 17 (score_kernel<true>, one empty
    category) agree within 1e-12.  score_kernel<true> at C = 17, 40, 120, 255 gives the same bits: an empty row adds
    fma(0, 0, acc) = acc and + 0 to the norms, the staged and the unstaged branch read the same keys, and nothing
    else depends on C.  small: staged at every C but 255 (one warp from C = 120 on).  large: pairs above 2 048 keys
    read from global memory next to staged ones at C = 17 and 40; at C = 120 the stage no longer fits and the whole
    launch reads from global memory, at C = 255 there never is a stage."""
    clouds, anchors, n = _small_set16() if which == "small" else _large_set(16, 310)
    pairs = np.stack([np.arange(n), n + np.arange(n)], axis=1)
    want = None
    res, regimes = {}, {}
    for C in (16, 17, 40, 120, 255):
        op = _params(gpu_ctx, oracle_mod, C, WF1, None, HELL2)
        s = _Set(gpu_ctx, clouds, anchors, 10.0)
        if want is None:
            want, counts = _oracle(oracle_mod, op, s, s, pairs, debug=True)
            assert np.all(counts.sum(axis=(0, 1))[:16] > 0)
        route = _route(C, HELL2, None, WF1, s, s)
        res[C] = _score(gpu_ctx, s, s, pairs, route, label=f"b {which}")
        assert_scores_close(res[C], want)
        regimes[C] = route
        if C >= 17:
            sz = s.sizes[pairs[:, 0]] + s.sizes[pairs[:, 1]]
            regimes[C] = dict(route["generic"], staged_pairs=int(np.sum(np.vectorize(_pad)(s.sizes[pairs[:, 0]]) +
                                                                        np.vectorize(_pad)(s.sizes[pairs[:, 1]])
                                                                        <= route["generic"]["stage_cap"])),
                              largest_pair=int(sz.max()))
        s.close()
    print(f"b {which}: {regimes}")
    g = {C: regimes[C] for C in (17, 40, 120, 255)}
    if which == "small":
        assert regimes[16]["launches"] == 1 and g[17]["warps"] > 1 and g[17]["stage_cap"] > 0
        assert g[120]["warps"] == 1 and g[120]["stage_cap"] > 0 and g[120]["staged_pairs"] == n
    else:
        assert regimes[16]["launches"] == 2 and g[17]["largest_pair"] > STAGE_MAX
        for C in (17, 40):
            assert g[C]["stage_cap"] == STAGE_MAX and 0 < g[C]["staged_pairs"] < n
        assert g[40]["warps"] > 1 and g[120]["stage_cap"] == 0
    assert g[255]["stage_cap"] == 0 and g[255]["warps"] == 1 and g[255]["smem"] == 195856
    assert np.abs(res[16] - res[17]).max() <= ROUTE_TOL
    for C in (40, 120, 255):
        assert np.array_equal(res[C], res[17]), f"C = {C} differs from C = 17"


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True], ids=["unit", "weighted"])
def test_empty_rows_of_the_fast_kernel_add_nothing(gpu_ctx, oracle_mod, weighted):
    """A 3-category structure scored at C = 3 and 8 (score_fast_kernel<8, ...>) and at C = 9 and 16 (<16, ...>): the
    rows of the categories that never occur hold zero counts, which add fma(0, 0, D) = D, 0 to the mismatch count and
    fma(w, 0, N) = N to the weighted totals, so within one row count the scores are bit-identical.  (Weights of the
    categories 0..2 are the same at every C.)"""
    base = synth.gen(400, 100, 4, 3)
    partner = synth.partner(base, 1.0, 4000)
    anchors = np.arange(0, base.n, 2, dtype=np.uint32)
    n = len(anchors)
    pairs = np.stack([np.arange(n), n + np.arange(n)], axis=1)
    sets = [([base, partner], np.r_[_anchors(0, anchors), _anchors(1, anchors)], 10.0)]
    res = {}
    for C in (3, 8, 9, 16):
        weights = np.r_[[0.45, 2.6, 1.3], _cat_weights(C)[3:]] if weighted else None
        cp = 8 if C <= 8 else 16
        expect = {"launches": 1, "fast": f"score_fast_kernel<{cp}, true, {str(weighted).lower()}>"}
        res[C], _, _, built, _ = _case(gpu_ctx, oracle_mod, C, HELL2, weights, WF1, sets, pairs, label="b 3 categories",
                                    expect=expect)
        _close(built)
    assert np.array_equal(res[3], res[8])
    assert np.array_equal(res[9], res[16])


# ---- c. large category counts against the oracle ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C", [17, 64, 120, 134, 255])
def test_large_category_counts(gpu_ctx, oracle_mod, C):
    """score_kernel at C = 17 (staged, several warps), 64 and 120 (staged, one warp), 134 and 255 (no stage fits, one
    warp): environments of 40 - 250 members, categories uniform over C, C - 1 inside environments.  Every statistical
    distance, with unit weights and one weight function (W-keyed store) and with uneven weights and three weight
    functions chosen per pair (distance-keyed)."""
    base = synth.gen(500 + C, 200, 4, C)
    partner = synth.partner(base, 1.0, 5000 + C)
    anchors = np.arange(1, base.n, 8, dtype=np.uint32)
    n = len(anchors)
    pairs = np.stack([np.arange(n), n + (np.arange(n) + 3) % n], axis=1)
    wf_idx = (np.arange(n) % 3).astype(np.uint32)
    sets = [([base, partner], np.r_[_anchors(0, anchors), _anchors(1, anchors)], 12.0)]
    staged, warps = score_state_bytes(C) + 8 * 1278 <= SCORE_BUDGET, 1 if C >= 67 else None
    for k, sd in enumerate(SDS):
        for weights, wfs, idx in ((None, WF1, None), (_cat_weights(C), WFS3, wf_idx)):
            got, want, route, built, counts = _case(gpu_ctx, oracle_mod, C, sd, weights, wfs, sets, pairs, idx, "c")
            g = route["generic"]
            assert (g["stage_cap"] > 0) == staged and (warps is None or g["warps"] == warps)
            assert (C == 17) == (g["warps"] > 1)
            if k == 0 and weights is None:
                s = built[0]
                assert 30 <= s.sizes.min() and s.max <= 320
                anchor_last = np.stack([base.cat[anchors] == C - 1,
                                        partner.cat[anchors][(np.arange(n) + 3) % n] == C - 1], axis=1)
                assert (counts[:, :, C - 1] - anchor_last).max() > 0, "category C - 1 never inside an environment"
            _close(built)


@pytest.mark.gpu
def test_staged_and_unstaged_pairs_in_one_generic_launch(gpu_ctx, oracle_mod):
    """C = 17, generalised Hellinger (score_kernel<false>), uneven weights, three weight functions per pair: pairs of
    up to 2 048 keys staged, larger ones read from global memory, in one launch."""
    clouds, anchors, n = _large_set(17, 320)
    pairs = np.stack([np.arange(n), n + np.arange(n)], axis=1)
    wf_idx = (np.arange(n) % 3).astype(np.uint32)
    sd = SDS[1]
    expect = {"launches": 1, "stage_cap": STAGE_MAX}
    _, want, route, built, _ = _case(gpu_ctx, oracle_mod, 17, sd, _cat_weights(17), WFS3, [(clouds, anchors, 10.0)],
                                  pairs, wf_idx, "c mixed", expect)
    s = built[0]
    keys = np.vectorize(_pad)(s.sizes[pairs[:, 0]]) + np.vectorize(_pad)(s.sizes[pairs[:, 1]])
    print(f"c mixed: {np.sum(keys <= STAGE_MAX)} staged pairs, {np.sum(keys > STAGE_MAX)} from global memory")
    assert 0 < np.sum(keys <= STAGE_MAX) < n and route["generic"]["warps"] > 1
    assert np.all(np.isfinite(want))
    _close(built)


@pytest.mark.gpu
def test_category_255_is_unknown_at_255_categories(gpu_ctx, oracle_mod):
    """C = 255: a member of category 255 (as u16) inside an environment raises status 3 from the scoring launch; the
    same data with 254 in its place scores like the oracle."""
    C = 255
    base = synth.gen(600, 60, 4, C - 1)
    partner = synth.partner(base, 1.0, 6000)
    anchors = np.arange(0, base.n, 4, dtype=np.uint32)
    n = len(anchors)
    pairs = np.stack([np.arange(n), n + np.arange(n)], axis=1)
    d = np.linalg.norm(partner.xyz - partner.xyz[anchors[3]], axis=1)
    member = int(np.flatnonzero((d > 0) & (d < 5.0))[0])
    assert member not in anchors
    for cat, status in ((255, 3), (254, 0)):
        partner.cat[member] = cat
        op = _params(gpu_ctx, oracle_mod, C, WF1, None, HELL2)
        s = _Set(gpu_ctx, [base, partner], np.r_[_anchors(0, anchors), _anchors(1, anchors)], 10.0)
        route = _route(C, HELL2, None, WF1, s, s)
        if status:
            before = gpu_ctx.launch_count
            with pytest.raises(_capi.LocoHDError) as ei:
                gpu_ctx.score_pairs(s.env, s.env, pairs.astype(np.uint32))
            assert ei.value.status == status and gpu_ctx.launch_count - before == route["launches"]
        else:
            got = _score(gpu_ctx, s, s, pairs, route, label="c category 254")
            assert_scores_close(got, _oracle(oracle_mod, op, s, s, pairs))
        s.close()


# ---- d. the split between the fast kernel and the second pass --------------------------------------------------------
def _split_ensemble():
    """A dense ball (90 % category 0; environments of 700 - 2 300 members at threshold 10 A) and a sparse cloud
    (environments of 20 - 100): the mean environment is large enough that the stage reaches its 2 048-key cap from
    the members alone, the largest environments are larger than that, so the tables are sized to the stage."""
    ball = _ball(710, 2400, 7, 10.0, first_share=0.93)
    sparse = _sparse_cloud(711, 2000, 45.0, 7)
    d = np.linalg.norm(sparse.xyz[:, None, :] - sparse.xyz[None, :, :], axis=2)
    sizes = (d < 10.0).sum(axis=1)
    sparse_anchors = np.flatnonzero((sizes >= 20) & (sizes <= 100))[::20].astype(np.uint32)
    return [ball, sparse], np.r_[_anchors(0, _by_radius(ball, 10)), _anchors(1, sparse_anchors)]


def _pick(sizes, is_ball, target, a_ball, b_ball, exclude=()):
    """The first pair (i, j) of environments with pad(M_i) + pad(M_j) == target, i from the ball or not, j too."""
    p = np.vectorize(_pad)(sizes)
    for i in np.flatnonzero(is_ball == a_ball):
        for j in np.flatnonzero((is_ball == b_ball) & (p == target - p[i])):
            if (i, j) not in exclude and i != j:
                return int(i), int(j)
    return None


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["unit", "weighted", "three-wfs"])
def test_stage_split(gpu_ctx, oracle_mod, monkeypatch, variant):
    """pad_max > 2 048 and the stage at its cap (2 048 keys, tables of 2 048 entries): pairs well below the stage,
    at exactly Ma_pad + Mb_pad == stage (the fast kernel scores them: a ball environment of ~2 000 members, over 90 %
    of them one category, with a sparse one, and two ball environments), at stage + 2 and far above (the second
    score_kernel pass).  Two launches, every score like the oracle.  The staged pairs again from sets built only from
    their anchors - the pairs below the stage from two sets with pad_max <= 1 024 (stage == pad_max), each boundary
    pair from two sets of one environment (stage == pad_max == 2 048): other stages and table sizes, the same bits.
    Every set here is built by the multi-kernel gather, which the first one takes anyway (environments above 1 024
    members): the fused gather evaluates W(d) of a W-keyed store with its own square root and weight-function forms,
    which may differ from the multi-kernel gather's in the last bit (the tests of the gathers compare distances)."""
    C = 7
    monkeypatch.setenv("LOCOHD_LEGACY_GATHER", "1")
    weights = _cat_weights(C) if variant == "weighted" else None
    wfs = WFS3 if variant == "three-wfs" else WF1
    clouds, anchors = _split_ensemble()
    op = _params(gpu_ctx, oracle_mod, C, wfs, weights, HELL2)
    s = _Set(gpu_ctx, clouds, anchors, 10.0)
    route = _route(C, HELL2, weights, wfs, s, s)
    stage = route["stage"]
    ball = anchors[:, 0] == 0
    sz = s.sizes
    assert route["pad_max"] > 1024 and stage < route["pad_max"]
    assert stage == STAGE_MAX and route["table_n"] == STAGE_MAX and route["launches"] == 2
    assert 20 <= sz[~ball].min() and sz[~ball].max() <= 100 and sz[ball].max() + 2 > STAGE_MAX
    edge_sparse = _pick(sz, ball, stage, True, False)
    edge_ball = _pick(sz, ball, stage, True, True)
    above2 = _pick(sz, ball, stage + 2, True, False) or _pick(sz, ball, stage + 2, True, True)
    assert edge_sparse and edge_ball and above2, "no pair at the boundary"
    bi, si = np.flatnonzero(ball), np.flatnonzero(~ball)
    big = bi[np.argsort(sz[bi], kind="stable")]
    below = [(si[1], si[2]), (big[0], si[3]), (big[1], si[4])]
    far = [(big[-1], big[-2]), (big[-3], si[0])]
    pairs = np.array(below + [edge_sparse, edge_ball, above2] + far, dtype=np.int64)
    keys = np.vectorize(_pad)(sz[pairs[:, 0]]) + np.vectorize(_pad)(sz[pairs[:, 1]])
    print(f"d {variant}: stage={stage} pair keys={keys.tolist()}")
    assert np.all(keys[:3] <= 1024) and keys[3] == keys[4] == stage and keys[5] == stage + 2
    assert np.all(keys[6:] > stage + 100)
    wf_idx = (np.arange(len(pairs)) % 3).astype(np.uint32) if len(wfs) > 1 else None
    got = _score(gpu_ctx, s, s, pairs, route, wf_idx, f"d {variant}")
    want, counts = _oracle(oracle_mod, op, s, s, pairs, wf_idx, debug=True)
    assert_scores_close(got, want)
    a_edge = counts[3, 0]
    print(f"d {variant}: boundary pair sizes {sz[pairs[3]].tolist()}, category 0 holds {a_edge[0]} of {a_edge.sum()}")
    assert a_edge[0] >= 0.9 * a_edge.sum() and a_edge[0] > 1024
    # the staged pairs from sets of their own anchors
    for group in ([0, 1, 2], [3], [4]):
        g = pairs[group]
        sa = _Set(gpu_ctx, clouds, anchors[g[:, 0]], 10.0)
        sb = _Set(gpu_ctx, clouds, anchors[g[:, 1]], 10.0)
        assert np.array_equal(sa.sizes, sz[g[:, 0]]) and np.array_equal(sb.sizes, sz[g[:, 1]])
        r2 = _route(C, HELL2, weights, wfs, sa, sb)
        assert r2["launches"] == 1 and r2["stage"] == r2["pad_max"]
        assert (r2["stage"], r2["table_n"]) != (stage, route["table_n"]) or len(g) == 1
        sub = np.stack([np.arange(len(g))] * 2, axis=1)
        again = _score(gpu_ctx, sa, sb, sub, r2, None if wf_idx is None else wf_idx[group], f"d {variant} own sets")
        assert np.array_equal(again, got[group]), f"pairs {group}"
        sa.close()
        sb.close()
    s.close()


# ---- e. gradients at large C -----------------------------------------------------------------------------------------
def _grad_close(got, want, tol):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    err = float(np.abs(got - want).max()) if want.size else 0.0
    assert err <= tol * scale, f"max |diff| = {err} (scale {scale})"


GRAD_SDS = {17: gr.SDS["Kullback-Leibler"], 64: gr.SDS["Renyi"], 255: gr.SDS["Hellinger-e"]}


@pytest.mark.gpu
@pytest.mark.parametrize("C", [17, 64, 255])
def test_gradients_at_large_category_counts(gpu_ctx, oracle_mod, C):
    """score_grad_kernel<kCoords> (from_primitives_grad) and <kEntries> (from_rows_grad), one warp of
    grad_state_bytes(C) per CTA from C = 67 on, against the CPU references on tie-free cases, with uneven category
    weights and C - 1 in the data; Hellinger-2 and one other distance."""
    wf = gr.WFS["kumaraswamy"]
    for sd in (gr.SDS["Hellinger"], GRAD_SDS[C]):
        op = _params(gpu_ctx, oracle_mod, C, [wf], _cat_weights(C), sd)
        A, B, anchors = gr.tie_free_case(700 + C, [wf], C=C)
        A[1][1], B[1][4] = C - 1, C - 1
        print(f"e C={C} {sd}: grad warps={max(1, min(8, SCORE_BUDGET // grad_state_bytes(C)))} "
              f"smem={grad_state_bytes(C) * max(1, min(8, SCORE_BUDGET // grad_state_bytes(C)))}")
        before, tiles = gpu_ctx.launch_count, gpu_ctx.tile_launches
        plain = gpu_ctx.from_primitives(*A, *B, anchors, gr.THRESHOLD)
        n_plain = gpu_ctx.launch_count - before
        before = gpu_ctx.launch_count
        s, ga, gb = gpu_ctx.from_primitives_grad(*A, *B, anchors, gr.THRESHOLD)
        assert gpu_ctx.launch_count - before == n_plain and gpu_ctx.tile_launches == tiles
        assert np.abs(s - plain).max() <= ROUTE_TOL
        assert_scores_close(s, oracle_mod.from_primitives(op, *A, *B, anchors, gr.THRESHOLD))
        _, ra, rb = gr.from_primitives_grad(oracle_mod, op, *A, *B, anchors, gr.THRESHOLD)
        _grad_close(ga, ra, GRAD_TOL)
        _grad_close(gb, rb, GRAD_TOL)

        xa, ca, xb, cb = rr.tie_free_clouds(800 + C, gr.kinks([wf]), n=12, C=C)
        ca[2], cb[5] = C - 1, C - 1
        ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
        before = gpu_ctx.launch_count
        ea, eb = gpu_ctx.envset_from_rows(ta, ca), gpu_ctx.envset_from_rows(tb, cb)
        plain = gpu_ctx.score_pairs(ea, eb, np.stack([np.arange(12)] * 2, axis=1).astype(np.uint32))
        n_plain = gpu_ctx.launch_count - before
        ea.close(); eb.close()
        before = gpu_ctx.launch_count
        s, ga, gb = gpu_ctx.from_rows_grad(ta, ca, tb, cb)
        assert gpu_ctx.launch_count - before == n_plain and gpu_ctx.tile_launches == tiles
        assert np.abs(s - plain).max() <= ROUTE_TOL
        assert_scores_close(s, oracle_mod.from_dmxs(op, ca, cb, ta, tb))
        _, ra, rb = rr.from_rows_grad(oracle_mod, op, ta, ca, tb, cb)
        _grad_close(ga, np.array(ra), GRAD_TOL)
        _grad_close(gb, np.array(rb), GRAD_TOL)


# ---- f. category-count limits ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_anchor_lists_at_255_categories(gpu_ctx, oracle_mod):
    """The from_anchors walk (one thread, PMFs of 255 entries) with categories 0..254 all present."""
    C = 255
    rng = np.random.default_rng(901)
    for sd, weights in ((HELL2, None), (SDS[3], _cat_weights(C))):
        op = _params(gpu_ctx, oracle_mod, C, WFS3, weights, sd)
        seq_a = np.r_[rng.permutation(C), rng.integers(0, C, 45)].astype(np.uint16)
        seq_b = np.r_[rng.integers(0, C, 200), [C - 1, 0]].astype(np.uint16)
        da = np.r_[0.0, np.sort(rng.uniform(0.5, 13.0, len(seq_a) - 1))]
        db = np.r_[0.0, np.sort(rng.uniform(0.5, 13.0, len(seq_b) - 1))]
        for wf in range(3):
            before, tiles = gpu_ctx.launch_count, gpu_ctx.tile_launches
            got = gpu_ctx.score_anchor_lists(seq_a, da, seq_b, db, wf_idx=wf)
            assert gpu_ctx.launch_count - before == 3 and gpu_ctx.tile_launches == tiles   # two conversions, one walk
            want = oracle_mod.from_anchors(op, seq_a, seq_b, da, db, wf_idx=wf)
            print(f"f anchor lists C={C} {sd} wf={wf}: {got} vs {want}")
            assert_scores_close(got, want)


@pytest.mark.gpu
def test_category_count_limit_of_the_c_abi(fresh_ctx, oracle_mod):
    """set_params(255) succeeds; 256 categories: LOCOHD_ERR_UNSUPPORTED (102), and the context keeps working."""
    _params(fresh_ctx, oracle_mod, 255, WF1)
    with pytest.raises(_capi.LocoHDError) as ei:
        fresh_ctx.set_params(256, WF1)
    assert ei.value.status == 102
    op = _params(fresh_ctx, oracle_mod, 5, WF1)
    a = synth.gen(910, 40, 4, 5)
    b = synth.partner(a, 1.0, 911)
    anchors = np.stack([np.arange(0, a.n, 3)] * 2, axis=1).astype(np.uint32)
    got = fresh_ctx.from_primitives(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0)
    assert_scores_close(got, oracle_mod.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0))


def test_locohd_category_count_limit():
    """The drop-in class takes 255 category names and refuses 256 (no device is touched before the first score)."""
    import loco_hd

    loco_hd.LoCoHD([f"t{i}" for i in range(255)])
    with pytest.raises(ValueError):
        loco_hd.LoCoHD([f"t{i}" for i in range(256)])


# ---- CPU: the restated rules -----------------------------------------------------------------------------------------
def test_generic_kernel_regimes():
    """score_kernel's shape as C grows: a 2 048-key stage fits up to C = 111, any stage up to C = 133; two or more
    warps up to C = 66 without a stage; 195 856 bytes of shared memory at C = 255."""
    assert score_state_bytes(255) == 195856 and score_state_bytes(17) == 13072
    assert generic_launch(111, True, 4096)["stage_cap"] == STAGE_MAX
    assert generic_launch(112, True, 4096)["stage_cap"] == 0
    assert generic_launch(120, True, 1278)["stage_cap"] == 1278 and generic_launch(120, True, 1280)["stage_cap"] == 0
    assert generic_launch(133, True, 30)["stage_cap"] == 30 and generic_launch(134, True, 2)["stage_cap"] == 0
    assert generic_launch(66, True, 0)["warps"] == 2 and generic_launch(67, True, 0)["warps"] == 1
    assert generic_launch(17, True, 2048)["warps"] == 3 and generic_launch(40, True, 2048)["warps"] == 2
    assert generic_launch(255, False, 600) == {"kernel": "score_kernel<false>", "stage_cap": 0, "warps": 1,
                                               "smem": 195856}
    assert max(1, min(8, SCORE_BUDGET // grad_state_bytes(255))) == 1 and grad_state_bytes(255) == 195840


def test_fast_route_rules():
    """One launch while the largest pair is at most 1 024 keys; above that a stage of 1.5 (mean_a + mean_b) + 64 keys
    rounded to 64, at most 2 048 and pad_max, and a second pass for what it leaves; tables of min(max + 2, stage)."""
    r = pair_route(7, True, True, True, 500, 510, 300.0, 300.0)
    assert r["launches"] == 1 and r["stage"] == 1010 and r["table_n"] == 512
    r = pair_route(7, True, True, True, 2300, 2300, 900.0, 900.0)
    assert r["launches"] == 2 and r["stage"] == 2048 and r["table_n"] == 2048 and r["second"]["stage_cap"] == 0
    assert pair_route(16, True, False, False, 100, 100, 50.0, 50.0)["fast"] == "score_fast_kernel<16, false, true>"
    assert pair_route(17, True, True, True, 100, 100, 50.0, 50.0)["generic"]["kernel"] == "score_kernel<true>"
    assert pair_route(5, False, True, True, 100, 100, 50.0, 50.0)["generic"]["kernel"] == "score_kernel<false>"
    assert fast_stage(1100, 100.0, 100.0) == 384   # a stage below pad_max that depends on the mean
    with pytest.raises(AssertionError):
        pair_route(7, True, True, True, 600, 600, 100.0, 100.0)
