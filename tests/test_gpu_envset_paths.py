"""Which gather builds an environment set.  The fused gather and the multi-kernel gather give the same environments,
so the parity tests cannot tell them apart; these tests pin the route every call takes through the context's launch
counter and its per-group profile records (one record per bracketed launch group):

    count  the 1/16 sizing sample of the fused gather, or the upper-bound sizes of the multi-kernel gather
    fill   one per fused attempt (512- or 1 024-member instantiation), plus the multi-kernel fill
    scan   multi-kernel gather only
    sort   multi-kernel gather only

Each step builds the environments of one fresh structure (so its cells are built too) and checks the sizes of a sample
of anchors against the oracle.  Each test starts from a fresh context: the store-sizing history and the 512 / 1 024
hint are per context.
"""
import numpy as np
import pytest

from benchdata import synth
from helpers import random_cloud, set_both
from loco_hd_b200 import _capi

pytestmark = pytest.mark.gpu

GROUPS = ("count", "fill", "scan", "sort")


@pytest.fixture
def ctx():
    c = _capi.Context(0)
    yield c
    c.close()


def route(ctx, oracle_mod, op, S, anchors, threshold):
    """Builds the environments of `anchors` in S -> (records per group of GROUPS, launches).  Asserts the sizes of up
    to 8 anchors against the oracle."""
    anchors = np.ascontiguousarray(anchors, dtype=np.uint32)
    st = ctx.structure(*S)
    ctx.profile_read()
    ctx.profile_enable(True)
    launches = ctx.launch_count
    env = ctx.envset_build(st, anchors, threshold)
    launches = ctx.launch_count - launches
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    off = np.empty(len(anchors) + 1, np.uint64)
    ctx._check(ctx.lib.locohd_envset_dump(ctx.h, env.h, _capi._p(off), None, None, None))
    env.close(); st.close()
    sizes = np.diff(off).astype(np.int64)
    for p in np.unique(np.linspace(0, len(anchors) - 1, 8).astype(int)):
        idx, _, _ = oracle_mod.environment(op, S[0], S[1], S[2], int(anchors[p]), threshold)
        assert sizes[p] == len(idx), f"environment size of anchor {p}"
    return {g: prof[g][1] for g in GROUPS}, launches


def expect(count, fill, scan, sort):
    return dict(count=count, fill=fill, scan=scan, sort=sort)


def protein(threshold):
    """3 200 primitives in 400 residues; all of them anchors (within the 32 768 bound: the store is sized by it)."""
    a = synth.gen(31, 400, 8, 7)
    return (a.xyz, a.cat, a.tag), np.arange(a.n), threshold


def between_512_and_1024():
    """synth.gen(53, 500, 8, 7) at 14.5 A: environments of 300-900 members."""
    a = synth.gen(53, 500, 8, 7)
    return (a.xyz, a.cat, a.tag), np.arange(a.n), 14.5


def cloud_40000(extent):
    """40 000 anchors (above the 32 768 bound: the store is sized by a sample or by the history) in a cube of side
    2 * extent at 10 A: about 12 members at extent 120, about 280 at extent 42."""
    n = 40000
    cat = np.random.default_rng(31).integers(0, 5, n).astype(np.uint16)
    xyz = np.random.default_rng(7 if extent > 100 else 8).uniform(-extent, extent, (n, 3))
    return (xyz, cat, np.arange(n, dtype=np.uint32)), np.arange(n), 10.0


def check_steps(ctx, oracle_mod, op, steps):
    for label, (S, anchors, threshold), want in steps:
        got = route(ctx, oracle_mod, op, S, anchors, threshold)
        assert got == want, label


def test_small_call_is_sized_by_the_bound(ctx, oracle_mod):
    op = set_both(ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    check_steps(ctx, oracle_mod, op, [
        ("protein at 8 A", protein(8.0), (expect(0, 1, 0, 0), 7)),
    ])


def test_store_sizing_by_sample_and_by_history(ctx, oracle_mod):
    """A first large call samples the sizes; a second call of the same shape takes the store size that worked then.
    When the same shape comes with much larger environments, the history-sized store overflows: the call is redone
    with a sampled size, which is then remembered in turn."""
    op = set_both(ctx, oracle_mod, 5, [("uniform", (3.0, 10.0))], tag_rule={"accept_same": False})
    check_steps(ctx, oracle_mod, op, [
        ("sparse, first call", cloud_40000(120.0), (expect(1, 1, 0, 0), 8)),
        ("sparse again", cloud_40000(120.0), (expect(0, 1, 0, 0), 7)),
        ("dense: the history-sized store overflows, then a sample", cloud_40000(42.0), (expect(1, 2, 0, 0), 9)),
        ("dense again", cloud_40000(42.0), (expect(0, 1, 0, 0), 7)),
    ])


def test_cap_hint_goes_up_and_comes_back_down(ctx, oracle_mod):
    """Environments beyond 512 members: the 512-member attempt reports them and the 1 024-member one builds the set;
    the context then starts with 1 024, until a 1 024 run sees no environment above 384 members."""
    op = set_both(ctx, oracle_mod, 7, [("uniform", (3.0, 14.0))], tag_rule={"accept_same": False})
    check_steps(ctx, oracle_mod, op, [
        ("512-1024 members, first call", between_512_and_1024(), (expect(0, 2, 0, 0), 8)),
        ("512-1024 members again: starts at 1024", between_512_and_1024(), (expect(0, 1, 0, 0), 7)),
        ("small environments at 1024: the hint drops", protein(8.0), (expect(0, 1, 0, 0), 7)),
        ("512-1024 members: starts at 512 again", between_512_and_1024(), (expect(0, 2, 0, 0), 8)),
    ])


def test_environments_above_1024_members_fall_back(ctx, oracle_mod):
    """Environments of 2 600 members have more candidates than the row-start bitmap of the 512-member attempt covers:
    that attempt reports an overflow other than the cap, so the call goes to the multi-kernel gather at once and the
    hint stays at 512.  Environments of 1 500 members fit the bitmap: 512, then 1024, then the multi-kernel gather."""
    rng = np.random.default_rng(10)
    big = random_cloud(rng, 2600, 6, extent=20.0)
    mid = random_cloud(rng, 1500, 6, extent=20.0)
    op = set_both(ctx, oracle_mod, 6, [("hyper_exp", (1.0, 0.05))])
    check_steps(ctx, oracle_mod, op, [
        ("2600 members", (big, np.arange(0, 2600, 65), 1000.0), (expect(1, 2, 1, 1), 13)),
        ("1500 members", (mid, np.arange(0, 1500, 65), 1000.0), (expect(1, 3, 1, 1), 13)),
    ])


def test_threshold_beyond_the_fused_range_falls_back(ctx, oracle_mod):
    rng = np.random.default_rng(9)
    S = random_cloud(rng, 200, 4)
    op = set_both(ctx, oracle_mod, 4)
    check_steps(ctx, oracle_mod, op, [
        ("r^2 >= 1e30", (S, np.arange(0, 200, 3), 1.0e16), (expect(1, 1, 1, 1), 8)),
    ])


def test_legacy_gather_switch(ctx, oracle_mod, monkeypatch):
    monkeypatch.setenv("LOCOHD_LEGACY_GATHER", "1")
    op = set_both(ctx, oracle_mod, 7, tag_rule={"accept_same": False})
    check_steps(ctx, oracle_mod, op, [
        ("protein at 8 A", protein(8.0), (expect(1, 1, 1, 1), 12)),
    ])
