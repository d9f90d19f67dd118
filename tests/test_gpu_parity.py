"""GPU parity tests: the CUDA path, called through the C ABI (loco_hd_b200._capi -> include/locohd_b200.h),
against the CPU oracle on the same inputs.  Bars (BASELINE.json north_star): neighbour lists and category counts
bit-exact; per-anchor scores within 1e-9 absolute.

Known answers come from the reference's own tests:
  /root/reference/tests/test_locohd.py:27-52, tests/test_tag_pairing_rule.py:100-157, tests/test_wfs.py:8-138.
"""
import numpy as np
import pytest

from benchdata import synth
from helpers import (SCORE_TOL, assert_scores_close, canonical_env, check_from_primitives, random_cloud,
                     set_both)

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- known answers
def test_from_anchors_known_answers(gpu_ctx, oracle_mod):
    # tests/test_locohd.py:30-40 (uniform [0, 4], categories O A B C)
    op = set_both(gpu_ctx, oracle_mod, 4, [("uniform", (0.0, 4.0))])
    seq = [0, 1, 2, 3]
    v1 = gpu_ctx.score_anchor_lists(seq, [0., 1., 2., 3.], seq, [0., 1., 1., 1.])
    v2 = gpu_ctx.score_anchor_lists(seq, [0., 1., 1., 1.], seq, [0., 1., 2., 3.])
    assert v1 == pytest.approx(0.2268, abs=5e-5) and v2 == pytest.approx(0.2268, abs=5e-5)
    assert abs(v1 - oracle_mod.from_anchors(op, seq, seq, [0., 1., 2., 3.], [0., 1., 1., 1.])) < SCORE_TOL
    # tests/test_locohd.py:42-52 (kumaraswamy [3, 10, 2, 5])
    op = set_both(gpu_ctx, oracle_mod, 3, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))])
    v = gpu_ctx.score_anchor_lists([0, 1, 0, 2], [0., 1., 5., 9.], [0, 2], [0., 7.])
    assert v == pytest.approx(0.4979, abs=5e-5)
    assert abs(v - oracle_mod.from_anchors(op, [0, 1, 0, 2], [0, 2], [0., 1., 5., 9.], [0., 7.])) < SCORE_TOL


NINE = dict(
    xyz=np.array([[0, 0, 0], [0, 1, 0], [2, 0, 0], [2, 2, 0], [1, 2, 0], [1, 3, 0], [3, 2, 0], [3, 3, 0], [2, 1, 0]],
                 dtype=np.float64),
    cat=np.array([0, 0, 0, 0, 1, 1, 1, 1, 2], dtype=np.uint16),
    anchors=[(0, 3), (4, 5), (0, 4), (0, 8), (4, 8)],
)


def test_tag_rule_inside_scoring(gpu_ctx, oracle_mod):
    # tests/test_tag_pairing_rule.py:100-157: tags = residue (= category) ids, uniform [1, 1.001], threshold 1.002
    S = (NINE["xyz"], NINE["cat"], NINE["cat"].astype(np.uint32))
    op = set_both(gpu_ctx, oracle_mod, 3, [("uniform", (1.0, 1.001))], tag_rule={"accept_same": True})
    got, _ = check_from_primitives(gpu_ctx, oracle_mod, op, S, S, NINE["anchors"], 1.002)
    assert np.allclose(got, [0., 0., 1., 1., 1.], atol=1e-15, rtol=0)
    op = set_both(gpu_ctx, oracle_mod, 3, [("uniform", (1.0, 1.001))], tag_rule={"accept_same": False})
    got, _ = check_from_primitives(gpu_ctx, oracle_mod, op, S, S, NINE["anchors"], 1.002)
    assert np.allclose(got, [0.7071, 0.5412, 0.5412, 0.4284, 0.6501], atol=5e-5, rtol=0)


def test_tag_pair_lists(gpu_ctx, oracle_mod):
    rng = np.random.default_rng(11)
    A = random_cloud(rng, 300, 5, extent=12.0, n_tags=6)
    B = random_cloud(rng, 280, 5, extent=12.0, n_tags=6)
    anchors = [(i, i) for i in range(0, 280, 3)]
    pairs = [(0, 1), (0, 2), (1, 2), (3, 3), (5, 0)]
    for accepted in (True, False):
        for ordered in (True, False):
            rule = {"tag_pairs": pairs, "accepted_pairs": accepted, "ordered": ordered}
            op = set_both(gpu_ctx, oracle_mod, 5, tag_rule=rule)
            check_from_primitives(gpu_ctx, oracle_mod, op, A, B, anchors, 9.0)


# ------------------------------------------------------------------------------- BASELINE.json configurations
def test_config1_coarse_grained_pair(gpu_ctx, oracle_mod):
    a, b = synth.config1()
    anchors = [(i, i) for i in range(0, a.n, a.k)]
    for rule in ({"accept_same": False}, None):
        op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0))], tag_rule=rule)
        got, ref = check_from_primitives(gpu_ctx, oracle_mod, op, (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag),
                                         anchors, 10.0)
        assert len(got) == 150


def test_config2_all_atom_pair_kumaraswamy(gpu_ctx, oracle_mod):
    a, b = synth.config2()
    anchors = [(i, i) for i in range(a.n)]
    op = set_both(gpu_ctx, oracle_mod, 7, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule={"accept_same": False})
    got, ref = check_from_primitives(gpu_ctx, oracle_mod, op, (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag),
                                     anchors, 10.0)
    assert len(got) == 10000 and np.all(got >= 0) and np.all(got <= 1)


def test_identical_structures_score_exactly_zero(gpu_ctx, oracle_mod):
    f0 = synth.config4_frame0()
    op = set_both(gpu_ctx, oracle_mod, 8, tag_rule={"accept_same": False})
    anchors = np.stack([f0.centroid_anchors()] * 2, axis=1)
    S = (f0.xyz, f0.cat, f0.tag)
    got = gpu_ctx.from_primitives(*S, *S, anchors, 10.0)
    assert np.all(got == 0.0), f"max = {np.abs(got).max()}"


def test_f32_exact_coordinates(gpu_ctx, oracle_mod):
    a = synth.gen(21, 200, 8, 7, f32_exact=True)
    b = synth.partner(a, 1.0, 22, f32_exact=True)
    op = set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    check_from_primitives(gpu_ctx, oracle_mod, op, (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag),
                          [(i, i) for i in range(0, a.n, 5)], 10.0)


def test_far_from_origin_coordinates(gpu_ctx, oracle_mod):
    # the FP32 prefilter works on coordinates relative to the bounding box: a large offset must not change anything
    a = synth.gen(23, 150, 8, 7)
    b = synth.partner(a, 1.0, 24)
    shift = np.array([1.0e6, -2.0e6, 3.0e5])
    op = set_both(gpu_ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    check_from_primitives(gpu_ctx, oracle_mod, op, (a.xyz + shift, a.cat, a.tag), (b.xyz + shift, b.cat, b.tag),
                          [(i, i) for i in range(0, a.n, 7)], 10.0)


# ------------------------------------------------------------------- all weight functions / distances / weights
WFS = [
    ("hyper_exp", (1.0, 0.10051591793984666)),
    ("hyper_exp", (0.49, 0.86, 0.55, 0.13, 0.096, 0.157)),
    ("dagum", (1.7, 2.9, 11.0)),
    ("uniform", (2.5, 9.75)),
    ("kumaraswamy", (4.2, 13.1, 2.7, 6.3)),
    ("kumaraswamy", (3.0, 10.0, 2.0, 5.0)),
]
SDS = [
    ("Hellinger", (2.0,)),
    ("Hellinger", (3.4277149325231795,)),
    ("Kolmogorov-Smirnov", ()),
    ("Kullback-Leibler", (3.241633447825855,)),
    ("Renyi", (2.3, 0.7)),
    ("Renyi", (1.0, 0.5)),
    ("Renyi", (0.0, 0.5)),
    ("Renyi", (float("inf"), 0.5)),
]


@pytest.mark.parametrize("sd", SDS, ids=lambda s: f"{s[0]}{list(s[1])}")
def test_random_clouds_threshold_50(gpu_ctx, oracle_mod, sd):
    """Clouds of the reference's fixture generator (tests/generate_locohd_testcases.py:106-120: 50-300 points,
    uniform(-50, 50), 5 types, threshold 50, empty tags with the default rule)."""
    rng = np.random.default_rng(5)
    A = random_cloud(rng, 244, 5)
    B = random_cloud(rng, 160, 5)
    anchors = [(i, i) for i in range(160)]
    for wf in WFS:
        op = set_both(gpu_ctx, oracle_mod, 5, [wf], statistical_distance=sd)
        check_from_primitives(gpu_ctx, oracle_mod, op, A, B, anchors, 50.0, check_envs=(wf is WFS[0]))


def test_category_weights(gpu_ctx, oracle_mod):
    rng = np.random.default_rng(6)
    A = random_cloud(rng, 200, 4, extent=15.0)
    B = random_cloud(rng, 210, 4, extent=15.0)
    anchors = [(i, (3 * i) % 210) for i in range(200)]
    w = [0.5, 1.0, 2.25, 3.7]
    for sd in (("Hellinger", (2.0,)), ("Hellinger", (1.3,)), ("Kullback-Leibler", (0.01,))):
        op = set_both(gpu_ctx, oracle_mod, 4, category_weights=w, statistical_distance=sd)
        check_from_primitives(gpu_ctx, oracle_mod, op, A, B, anchors, 12.0)


def test_per_anchor_weight_functions(gpu_ctx, oracle_mod):
    rng = np.random.default_rng(7)
    A = random_cloud(rng, 150, 5, extent=14.0)
    B = random_cloud(rng, 150, 5, extent=14.0)
    anchors = [(i, i) for i in range(150)]
    wf_idx = rng.integers(0, len(WFS), size=150).astype(np.uint32)
    op = set_both(gpu_ctx, oracle_mod, 5, WFS)
    check_from_primitives(gpu_ctx, oracle_mod, op, A, B, anchors, 11.0, wf_idx=wf_idx, check_envs=False)


# ------------------------------------------------------------------ one-call upload routes (staged / copied per input)
def test_from_primitives_device_inputs(gpu_ctx, oracle_mod):
    """Every input of a one-call score already on the device (torch CUDA tensors passed as raw pointers): the inputs
    are copied one by one into the call's device block instead of travelling in the pinned staging buffer.  Same
    scores, bit for bit, as the same call with numpy inputs."""
    import torch

    a, b = synth.config1()
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0)), ("kumaraswamy", (3.0, 10.0, 2.0, 5.0))],
                  tag_rule={"accept_same": False})
    rng = np.random.default_rng(19)
    anchors = np.stack([rng.permutation(a.n)[:200], rng.permutation(b.n)[:200]], axis=1).astype(np.uint32)
    wf_idx = rng.integers(0, 2, len(anchors)).astype(np.uint32)
    host = gpu_ctx.from_primitives(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0, wf_idx=wf_idx)
    # unsigned arrays travel as signed torch tensors of the same bits
    arrays = (a.xyz, a.cat.view(np.int16), a.tag.view(np.int32), b.xyz, b.cat.view(np.int16), b.tag.view(np.int32),
              anchors.view(np.int32), wf_idx.view(np.int32))
    dev = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in arrays]
    torch.cuda.synchronize()
    ptr = [t.data_ptr() for t in dev]
    got = gpu_ctx.from_primitives(*ptr[:7], 10.0, wf_idx=ptr[7], n_a=a.n, n_b=b.n, n_pairs=len(anchors))
    assert np.array_equal(got, host)
    ref = oracle_mod.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0, wf_idx=wf_idx)
    assert_scores_close(got, ref)
    # the indices matter: weight function 0 for every pair gives other scores
    assert not np.array_equal(got, gpu_ctx.from_primitives(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0))


def test_from_primitives_above_the_staging_limit(gpu_ctx, oracle_mod):
    """A host call whose upload exceeds the 8 MB staging buffer (525 000 anchor pairs of 16 B) copies its inputs one
    by one into the call's device block.  Every pair fits the scoring stage and its arithmetic does not depend on the
    other pairs of the launch, so the scores equal, bit for bit, those of the same pairs in two staged calls."""
    a = synth.gen(41, 625, 8, 7)   # 5 000 primitives each
    b = synth.partner(a, 1.0, 42)
    A, B = (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag)
    op = set_both(gpu_ctx, oracle_mod, 7, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule={"accept_same": False})
    rng = np.random.default_rng(43)
    anchors = rng.integers(0, a.n, size=(525_000, 2)).astype(np.uint32)
    whole = gpu_ctx.from_primitives(*A, *B, anchors, 10.0)
    half = len(anchors) // 2
    parts = np.concatenate([gpu_ctx.from_primitives(*A, *B, anchors[:half], 10.0),
                            gpu_ctx.from_primitives(*A, *B, anchors[half:], 10.0)])
    assert np.array_equal(whole, parts)
    sample = np.sort(rng.choice(len(anchors), 2000, replace=False))
    assert_scores_close(whole[sample], oracle_mod.from_primitives(op, *A, *B, anchors[sample], 10.0))


# --------------------------------------------------------------------------------------------------- edge cases
def test_ties_duplicates_and_lattice(gpu_ctx, oracle_mod):
    # cubic lattice: many exactly equal distances inside and across environments; plus coincident points
    g = np.arange(7, dtype=np.float64) * 1.5
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    xyz = np.concatenate([xyz, xyz[:20]])  # 20 primitives coincide with others (distance exactly 0 to them)
    rng = np.random.default_rng(8)
    cat = rng.integers(0, 4, size=len(xyz)).astype(np.uint16)
    tag = rng.integers(0, 30, size=len(xyz)).astype(np.uint32)
    cat2 = rng.integers(0, 4, size=len(xyz)).astype(np.uint16)
    anchors = [(i, (i * 7) % len(xyz)) for i in range(len(xyz))]
    for rule in (None, {"accept_same": False}):
        op = set_both(gpu_ctx, oracle_mod, 4, [("uniform", (0.0, 6.0))], tag_rule=rule)
        check_from_primitives(gpu_ctx, oracle_mod, op, (xyz, cat, tag), (xyz, cat2, tag), anchors, 4.6)


def test_anchor_only_environments(gpu_ctx, oracle_mod):
    # threshold smaller than every contact: both environments hold just the anchor
    rng = np.random.default_rng(9)
    A = random_cloud(rng, 50, 3)
    op = set_both(gpu_ctx, oracle_mod, 3)
    got, _ = check_from_primitives(gpu_ctx, oracle_mod, op, A, A, [(0, 1), (2, 2), (5, 9)], 1e-3)
    assert got[1] == 0.0


@pytest.mark.parametrize("n,thr", [(700, 30.0), (2600, 1000.0), (5000, float("inf"))])
def test_large_environments(gpu_ctx, oracle_mod, n, thr):
    """Environment sizes beyond the 256/512 shared-memory classes, and beyond 2048 (global-memory sort)."""
    rng = np.random.default_rng(10)
    A = random_cloud(rng, n, 6, extent=20.0)
    B = random_cloud(rng, n - 17, 6, extent=20.0)
    anchors = [(i, i) for i in range(0, n - 17, max(1, n // 40))]
    op = set_both(gpu_ctx, oracle_mod, 6, [("hyper_exp", (1.0, 0.05))])
    check_from_primitives(gpu_ctx, oracle_mod, op, A, B, anchors, thr)


def test_category_counts_above_1024_in_the_fast_kernel(gpu_ctx, oracle_mod):
    """Hellinger-2 pairs whose environments fit the fast kernel's stage together (Ma + Mb <= 2 046) while one category
    of A holds more than 1 024 members: the kernel's sqrt and ratio tables must reach every such count and total.  A is
    a dense ball (environments of 1 300-1 600 members around its centre), B a sparse one (~300), both 90 % category 0;
    A + B hold 2 040 points, so no pair can exceed the bound."""
    rng = np.random.default_rng(1024)

    def ball(n):   # n points uniform in a ball of radius 10 around the origin, 90 % of them category 0
        d = rng.normal(size=(n, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        xyz = d * (10.0 * rng.random(n) ** (1.0 / 3.0))[:, None]
        return xyz, (rng.random(n) < 0.1).astype(np.uint16), np.zeros(n, np.uint32)

    A, B = ball(1650), ball(390)
    core_a = np.flatnonzero(np.linalg.norm(A[0], axis=1) < 2.5)
    core_b = np.flatnonzero(np.linalg.norm(B[0], axis=1) < 4.0)
    anchors = np.stack([core_a, core_b[np.arange(len(core_a)) % len(core_b)]], axis=1)
    op = set_both(gpu_ctx, oracle_mod, 2, [("uniform", (0.0, 10.0))])
    _, ref = check_from_primitives(gpu_ctx, oracle_mod, op, A, B, anchors, 10.0)
    sizes = ref["env_sizes"]
    assert sizes[:, 0].max() > 1100 and sizes.sum(axis=1).max() <= 2046
    assert ref["counts"][:, 0, 0].max() > 1024


def test_empty_anchor_list(gpu_ctx, oracle_mod):
    rng = np.random.default_rng(12)
    A = random_cloud(rng, 30, 3)
    set_both(gpu_ctx, oracle_mod, 3)
    got = gpu_ctx.from_primitives(*A, *A, np.zeros((0, 2), np.uint32), 10.0)
    assert len(got) == 0


def test_error_paths(gpu_ctx, oracle_mod):
    from loco_hd_b200._capi import LocoHDError, UNKNOWN_CATEGORY
    rng = np.random.default_rng(13)
    xyz, cat, tag = random_cloud(rng, 40, 3, extent=5.0)
    set_both(gpu_ctx, oracle_mod, 3)
    with pytest.raises(LocoHDError) as e:   # anchor index out of range (reference: panic at locohd.rs:521)
        gpu_ctx.from_primitives(xyz, cat, tag, xyz, cat, tag, [(0, 40)], 10.0)
    assert e.value.status == 8
    with pytest.raises(LocoHDError) as e:   # threshold <= 0: empty environments (reference: panic at locohd.rs:74)
        gpu_ctx.from_primitives(xyz, cat, tag, xyz, cat, tag, [(0, 0)], 0.0)
    assert e.value.status == 7
    with pytest.raises(LocoHDError):        # NaN threshold
        gpu_ctx.from_primitives(xyz, cat, tag, xyz, cat, tag, [(0, 0)], float("nan"))
    bad = cat.copy()
    bad[7] = UNKNOWN_CATEGORY
    with pytest.raises(LocoHDError) as e:   # unknown category inside an environment (pmf.rs:38-42)
        gpu_ctx.from_primitives(xyz, bad, tag, xyz, cat, tag, [(0, 0)], 100.0)
    assert e.value.status == 3
    # ... but not when no environment contains it
    far = xyz.copy()
    far[7] = [1e4, 1e4, 1e4]
    gpu_ctx.from_primitives(far, bad, tag, xyz, cat, tag, [(0, 0)], 20.0)
    nanxyz = xyz.copy()
    nanxyz[3, 1] = np.nan
    with pytest.raises(LocoHDError) as e:
        gpu_ctx.from_primitives(nanxyz, cat, tag, xyz, cat, tag, [(0, 0)], 10.0)
    assert e.value.status == 6
    # the context stays usable after an error
    assert len(gpu_ctx.from_primitives(xyz, cat, tag, xyz, cat, tag, [(0, 0)], 10.0)) == 1
    # from_anchors validation (locohd.rs:70-77)
    with pytest.raises(LocoHDError) as e:
        gpu_ctx.score_anchor_lists([0, 1], [0.0, 1.0, 2.0], [0], [0.0])
    assert e.value.status == 1
    with pytest.raises(LocoHDError) as e:
        gpu_ctx.score_anchor_lists([0, 1], [0.5, 1.0], [0], [0.0])
    assert e.value.status == 2
    # constructor-level validation (locohd.rs:305-346, weight_function.rs:31-89)
    for kwargs in (dict(n_categories=0), dict(n_categories=3, category_weights=[1.0, 0.0, 1.0]),
                   dict(n_categories=3, category_weights=[1.0, -1.0, 1.0]),
                   dict(n_categories=3, weight_functions=[("uniform", (1.0, 0.0))]),
                   dict(n_categories=3, weight_functions=[("hyper_exp", (1.0, 2.0, 3.0))]),
                   dict(n_categories=3, weight_functions=[("kumaraswamy", (3.0, 1.0, 2.0, 2.0))]),
                   dict(n_categories=3, weight_functions=[("dagum", (1.0, -2.0, 3.0))])):
        with pytest.raises(LocoHDError):
            gpu_ctx.set_params(**kwargs)


# ------------------------------------------------------------------------------------ from_anchors exact order
def test_from_anchors_random_lists_including_unsorted(gpu_ctx, oracle_mod):
    rng = np.random.default_rng(14)
    for trial in range(40):
        wf = WFS[trial % len(WFS)]
        sd = SDS[trial % len(SDS)]
        op = set_both(gpu_ctx, oracle_mod, 5, [wf], statistical_distance=sd)
        na, nb = rng.integers(1, 60, size=2)
        da = np.concatenate([[0.0], rng.uniform(0, 15, na - 1).round(1)])
        db = np.concatenate([[0.0], rng.uniform(0, 15, nb - 1).round(1)])
        if trial % 3:  # sorted (the documented use), else caller-ordered as the reference accepts it
            da.sort()
            db.sort()
        sa, sb = rng.integers(0, 5, na), rng.integers(0, 5, nb)
        got = gpu_ctx.score_anchor_lists(sa, da, sb, db)
        ref = oracle_mod.from_anchors(op, sa, sb, da, db)
        assert_scores_close(got, ref)


# ------------------------------------------------------------------------------------- from_dmxs / from_coords
@pytest.mark.parametrize("n", [37, 300, 700, 2300])
def test_from_coords_and_dmxs(gpu_ctx, oracle_mod, n):
    rng = np.random.default_rng(15)
    xa, ca, _ = random_cloud(rng, n, 5, extent=25.0)
    xb, cb, _ = random_cloud(rng, n, 5, extent=25.0)
    op = set_both(gpu_ctx, oracle_mod, 5, [("hyper_exp", (1.0, 0.08))])
    ea = gpu_ctx.envset_from_coords(xa, ca)
    eb = gpu_ctx.envset_from_coords(xb, cb)
    pairs = np.stack([np.arange(n)] * 2, axis=1).astype(np.uint32)
    got = gpu_ctx.score_pairs(ea, eb, pairs)
    ref = oracle_mod.from_coords(op, ca, cb, xa, xb)
    assert np.abs(got - ref).max() <= SCORE_TOL
    if n <= 700:
        # distance matrices with +inf entries (compare_ensembles.py:261-263 bans contacts that way)
        dm = lambda x: np.sqrt(((x[:, None, :] - x[None, :, :]) ** 2).sum(-1))
        ma, mb = dm(xa), dm(xb)
        ma[rng.random(ma.shape) < 0.05] = np.inf
        np.fill_diagonal(ma, 0.0)
        op = set_both(gpu_ctx, oracle_mod, 5, [("uniform", (3.0, 10.0))])
        ea2 = gpu_ctx.envset_from_rows(ma, ca)
        eb2 = gpu_ctx.envset_from_rows(mb, cb)
        got = gpu_ctx.score_pairs(ea2, eb2, pairs)
        ref = oracle_mod.from_dmxs(op, ca, cb, ma, mb)
        assert np.abs(got - ref).max() <= SCORE_TOL
        # the same matrices as ragged rows of equal length (the path of the Python API's from_dmxs): same store
        ea3 = gpu_ctx.envset_from_ragged_rows(ma, ca)
        eb3 = gpu_ctx.envset_from_ragged_rows(mb, cb)
        assert np.array_equal(gpu_ctx.score_pairs(ea3, eb3, pairs), got)
        for rect, ragged in ((ea2, ea3), (eb2, eb3)):
            for x, y in zip(rect.dump(), ragged.dump()):
                assert np.array_equal(x, y)
            rect.close(); ragged.close()


# ------------------------------------------------------------------------------------------------- leaf math
def test_weight_function_cdfs(gpu_ctx, oracle_mod):
    x = np.concatenate([[0.0, 1e-300, 0.5, 1.0, 3.0, 5.0, 9.999, 10.0, 10.001, 1e6, np.inf],
                        np.random.default_rng(16).uniform(0, 30, 200)])
    for name, params in WFS + [("dagum", (10.0, 5.0, 2.0)), ("uniform", (0.0, 1.0)), ("hyper_exp", (1.0, 1.0))]:
        got = gpu_ctx.wf_integral_points(name, params, x)
        ref = np.array([oracle_mod.wf_integral_point(name, params, float(v)) for v in x])
        assert np.abs(got - ref).max() <= 1e-13, name
    # tests/test_wfs.py known answers
    r = lambda n, p, a, b: np.diff(gpu_ctx.wf_integral_points(n, p, [a, b]))[0]
    assert r("hyper_exp", [1., 1.], 0., 1.) == pytest.approx(0.6321, abs=5e-5)
    assert r("hyper_exp", [3., 5., 2., 1 / 3., 1 / 5., 1 / 10.], 5., 10.) == pytest.approx(0.2100, abs=5e-5)
    assert r("dagum", [2., 5., 1.], 1., 3.) == pytest.approx(0.2262, abs=5e-5)
    assert r("dagum", [10., 5., 2.], 5., 10.) == pytest.approx(0.7480, abs=5e-5)
    assert r("uniform", [2., 16.], 5., 10.) == pytest.approx(0.3571, abs=5e-5)
    assert r("kumaraswamy", [5., 10., 2., 3.], 6.4, 6.7) == pytest.approx(0.0910, abs=5e-5)
    assert r("kumaraswamy", [5., 9., 7., 7.], 5., 7.) == pytest.approx(0.0534, abs=5e-5)


def test_statistical_distances(gpu_ctx, oracle_mod):
    rng = np.random.default_rng(17)
    p1 = rng.random((64, 6)); p1[rng.random(p1.shape) < 0.2] = 0.0; p1[:, 0] += 1e-3; p1 /= p1.sum(1, keepdims=True)
    p2 = rng.random((64, 6)); p2[rng.random(p2.shape) < 0.2] = 0.0; p2[:, 1] += 1e-3; p2 /= p2.sum(1, keepdims=True)
    for name, params in SDS:
        got = gpu_ctx.sd_run(name, params, p1, p2)
        ref = np.array([oracle_mod.sd_run(name, params, a, b) for a, b in zip(p1, p2)])
        ok = np.isfinite(ref)
        assert np.array_equal(np.isfinite(got), ok)
        assert np.abs(got[ok] - ref[ok]).max() <= 1e-12, name


# --------------------------------------------------------------------------------- batches and size-independent
def test_batch_jobs_match_single_calls(gpu_ctx, oracle_mod):
    """CASP-style batch (config 3 shape, reduced): one reference against several models through the env-set /
    job API must equal the one-call drop-in on every structure pair."""
    ref = synth.gen(5, 60, 9, 8, with_centroid=True)
    models = [synth.config3_model(ref, m) for m in range(5)]
    op = set_both(gpu_ctx, oracle_mod, 8, tag_rule={"accept_same": False})
    clouds = [ref] + models
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    st = gpu_ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]), np.concatenate([c.cat for c in clouds]),
                                np.concatenate([c.tag for c in clouds]))
    cent = ref.centroid_anchors()
    a_struct = np.repeat(np.arange(len(clouds), dtype=np.uint32), len(cent))
    a_prim = np.tile(cent, len(clouds))
    env = gpu_ctx.envset_build(st, a_prim, 10.0, anchor_struct=a_struct)
    jobs = np.array([(0, (m + 1) * len(cent), len(cent)) for m in range(len(models))],
                    dtype=[("a_first", "<u8"), ("b_first", "<u8"), ("n", "<u8")])
    scores, means = gpu_ctx.score_jobs(env, env, jobs, want_means=True)
    scores = scores.reshape(len(models), len(cent))
    anchors = np.stack([cent, cent], axis=1)
    for m, model in enumerate(models):
        single = gpu_ctx.from_primitives(ref.xyz, ref.cat, ref.tag, model.xyz, model.cat, model.tag, anchors, 10.0)
        assert np.array_equal(single, scores[m])
        cpu = oracle_mod.from_primitives(op, ref.xyz, ref.cat, ref.tag, model.xyz, model.cat, model.tag, anchors, 10.0)
        assert np.abs(cpu - scores[m]).max() <= SCORE_TOL
        assert means[m] == pytest.approx(scores[m].mean(), abs=1e-14)
    # means only (SURVEY 8(f) N4: what bench.py copies out for the full-size ensemble): same values, caller's buffer
    only = np.full(len(models), np.nan)
    none, same = gpu_ctx.score_jobs(env, env, jobs, want_scores=False, means_out=only)
    assert none is None and same is only
    assert np.array_equal(only, means)


def test_symmetry_and_permutation_invariance(gpu_ctx, oracle_mod):
    """Size-independent properties at a full BASELINE size (config 2, 10k primitives): swapping the structures
    and shuffling the primitive order leave every score unchanged (the latter bit-exactly only up to summation
    order, hence the 1e-12 bar); scores lie in [0, 1]."""
    a, b = synth.config2()
    set_both(gpu_ctx, oracle_mod, 7, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule={"accept_same": False})
    anchors = np.stack([np.arange(a.n, dtype=np.uint32)] * 2, axis=1)
    s_ab = gpu_ctx.from_primitives(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0)
    s_ba = gpu_ctx.from_primitives(b.xyz, b.cat, b.tag, a.xyz, a.cat, a.tag, anchors, 10.0)
    assert np.abs(s_ab - s_ba).max() <= 1e-12
    perm = np.random.default_rng(18).permutation(a.n)
    inv = np.empty_like(perm); inv[perm] = np.arange(a.n)
    anchors_p = np.stack([inv.astype(np.uint32), np.arange(a.n, dtype=np.uint32)], axis=1)
    s_p = gpu_ctx.from_primitives(a.xyz[perm], a.cat[perm], a.tag[perm], b.xyz, b.cat, b.tag, anchors_p, 10.0)
    assert np.abs(s_ab - s_p).max() <= 1e-12
    assert s_ab.min() >= 0.0 and s_ab.max() <= 1.0


# ------------------------------------------------------------------------------- fused gather vs multi-kernel gather
def _dump_env(ctx, S, anchors, thr):
    st = ctx.structure(*S)
    env = ctx.envset_build(st, anchors, thr, keep_indices=True)
    out = env.dump()
    env.close()
    st.close()
    return out


@pytest.mark.parametrize("case", ["protein10", "cloud50", "sparse_anchors", "inf_small", "f32"])
def test_fused_gather_matches_multi_kernel_gather(oracle_mod, case, monkeypatch):
    """env_fused_kernel (one warp per anchor: gather + exact test + register sort + packing) and the multi-kernel
    path (count / scan / fill / bucket sort) must produce the same environments: sizes, categories, distances and
    - up to the order inside groups of equal (distance, category) - primitive indices."""
    from loco_hd_b200 import _capi
    rng = np.random.default_rng(77)
    if case == "protein10":
        a = synth.gen(31, 400, 8, 7)
        S, anchors, thr, C = (a.xyz, a.cat, a.tag), np.arange(a.n, dtype=np.uint32), 10.0, 7
    elif case == "cloud50":
        S, anchors, thr, C = random_cloud(rng, 300, 5, n_tags=40), np.arange(300, dtype=np.uint32), 50.0, 5
    elif case == "sparse_anchors":
        a = synth.gen(33, 300, 9, 8)
        S, anchors, thr, C = (a.xyz, a.cat, a.tag), np.arange(0, a.n, 9, dtype=np.uint32)[::-1].copy(), 7.5, 8
    elif case == "inf_small":
        S, anchors, thr, C = random_cloud(rng, 200, 4), np.arange(0, 200, 3, dtype=np.uint32), float("inf"), 4
    else:
        a = synth.gen(35, 250, 8, 7, f32_exact=True)
        S, anchors, thr, C = (a.xyz, a.cat, a.tag), np.arange(a.n, dtype=np.uint32), 10.0, 7
    outs = []
    for legacy in ("0", "1"):
        monkeypatch.setenv("LOCOHD_LEGACY_GATHER", legacy)
        ctx = _capi.Context(0)
        ctx.set_params(C, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule={"accept_same": False})
        outs.append(_dump_env(ctx, S, anchors, thr))
        ctx.close()
    (off0, d0, c0, i0), (off1, d1, c1, i1) = outs
    assert np.array_equal(off0, off1)
    assert np.array_equal(d0, d1), "sorted distances differ"
    assert np.array_equal(c0, c1), "categories differ"
    for p in range(len(anchors)):
        a0, _ = canonical_env(i0[off0[p]:off0[p + 1]], d0[off0[p]:off0[p + 1]])
        a1, _ = canonical_env(i1[off1[p]:off1[p + 1]], d1[off1[p]:off1[p + 1]])
        assert np.array_equal(a0, a1), f"members differ for anchor {p}"


# ------------------------------------------------------------------------------- fused gather: geometry corner cases
def test_members_exactly_on_the_sphere_are_excluded(gpu_ctx, oracle_mod):
    """Integer lattice, threshold exactly 5: primitives at distance exactly 5 (3-4-5 and axis neighbours) sit on the
    strict `d2 < r2` boundary and on cell / row-pruning boundaries at the same time."""
    g = np.arange(-6, 7, dtype=np.float64)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    rng = np.random.default_rng(12)
    cat = rng.integers(0, 5, size=len(xyz)).astype(np.uint16)
    tag = np.arange(len(xyz), dtype=np.uint32)
    centre = int(np.flatnonzero((xyz == 0).all(axis=1))[0])
    anchors = [(centre, centre)] + [(int(i), int(i)) for i in rng.choice(len(xyz), 40, replace=False)]
    op = set_both(gpu_ctx, oracle_mod, 5, [("uniform", (1.0, 5.0))], tag_rule={"accept_same": False})
    _, ref = check_from_primitives(gpu_ctx, oracle_mod, op, (xyz, cat, tag), (xyz, cat, tag), anchors, 5.0)
    # the centre sees every lattice point with x^2 + y^2 + z^2 < 25 (itself included)
    assert ref["env_sizes"][0, 0] == int(((xyz ** 2).sum(axis=1) < 25).sum())


@pytest.mark.parametrize("shape", ["line", "plane", "point", "two_clusters", "f32_far"])
def test_degenerate_structures(gpu_ctx, oracle_mod, shape):
    """Flat, linear, single-point and widely separated structures: grids with one cell along some axes, enlarged
    cells, empty rows; every primitive an anchor, neighbour lists compared with the oracle."""
    rng = np.random.default_rng(13)
    n = 160
    if shape == "line":
        xyz = np.zeros((n, 3)); xyz[:, 0] = np.sort(rng.uniform(0, 300, n))
    elif shape == "plane":
        xyz = np.zeros((n, 3)); xyz[:, 1:] = rng.uniform(0, 40, (n, 2)); xyz[:, 0] = 7.25
    elif shape == "point":
        xyz = np.tile(np.array([[1.5, -2.5, 3.0]]), (n, 1))
    elif shape == "two_clusters":
        xyz = rng.normal(0, 4, (n, 3)); xyz[n // 2:] += np.array([5000.0, -3000.0, 800.0])
    else:
        xyz = (rng.uniform(-30, 30, (n, 3)) + np.array([9.0e4, 9.0e4, -9.0e4])).astype(np.float32).astype(np.float64)
    cat = rng.integers(0, 4, size=n).astype(np.uint16)
    tag = (np.arange(n) // 4).astype(np.uint32)
    anchors = [(i, (i * 3) % n) for i in range(n)]
    op = set_both(gpu_ctx, oracle_mod, 4, [("dagum", (3.0, 6.0, 2.0))], tag_rule={"accept_same": False})
    check_from_primitives(gpu_ctx, oracle_mod, op, (xyz, cat, tag), (xyz[::-1].copy(), cat, tag), anchors, 10.0)


def test_one_oversized_environment_falls_back(gpu_ctx, oracle_mod):
    """One dense blob (> 512 members around its anchors) next to an ordinary structure: the 512-member instantiation
    of the fused gather reports the overflow and the call is redone by the 1024-member one (and the context then
    starts with it; a later call with small environments goes back to 512) - same results as the oracle."""
    rng = np.random.default_rng(14)
    blob = rng.normal(0, 2.0, (700, 3))
    rest = rng.uniform(-40, 40, (600, 3)) + np.array([80.0, 0, 0])
    xyz = np.concatenate([blob, rest])
    cat = rng.integers(0, 6, size=len(xyz)).astype(np.uint16)
    tag = rng.integers(0, 200, size=len(xyz)).astype(np.uint32)
    anchors = [(i, i) for i in range(0, len(xyz), 13)]
    op = set_both(gpu_ctx, oracle_mod, 6, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule={"accept_same": False})
    _, ref = check_from_primitives(gpu_ctx, oracle_mod, op, (xyz, cat, tag), (xyz, cat, tag), anchors, 10.0)
    assert ref["env_sizes"].max() > 512
    # back to ordinary sizes on the same context
    a = synth.gen(51, 120, 8, 6)
    check_from_primitives(gpu_ctx, oracle_mod, op, (a.xyz, a.cat, a.tag), (a.xyz, a.cat, a.tag),
                          [(i, i) for i in range(0, a.n, 7)], 10.0)
    check_from_primitives(gpu_ctx, oracle_mod, op, (a.xyz, a.cat, a.tag), (a.xyz, a.cat, a.tag),
                          [(i, i) for i in range(0, a.n, 7)], 10.0)


def test_environments_between_512_and_1024_members(gpu_ctx, oracle_mod):
    """Protein-like structure at a 14.5 A threshold: environments of 300-900 members (fused gather, 1024-member
    instantiation, 32 keys per lane in the register sort)."""
    a = synth.gen(53, 500, 8, 7)
    b = synth.partner(a, 1.0, 54)
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 14.0))], tag_rule={"accept_same": False})
    _, ref = check_from_primitives(gpu_ctx, oracle_mod, op, (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag),
                                   [(i, i) for i in range(0, a.n, 9)], 14.5)
    assert 512 < ref["env_sizes"].max() <= 1024
