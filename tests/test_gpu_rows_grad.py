"""GPU tests of the gradients of from_dmxs and from_coords scores (locohd_from_rows_grad, locohd_from_coords_grad,
LoCoHD.from_dmxs_grad / from_coords_grad).

Scores must equal those of the plain calls (1e-12); gradients must equal those of the CPU reference in
tests/rows_grad_reference.py (1e-9 relative to max(1, max |g|)), whose own gradients are checked against finite
differences of the oracle in tests/test_rows_grad_oracle.py.  Both calls are deterministic: repeated calls are
byte-identical.
"""
import numpy as np
import pytest

import rows_grad_reference as rr
from benchdata import synth
from grad_reference import SDS, WFS, kinks
from helpers import set_both

pytestmark = pytest.mark.gpu

GRAD_TOL = 1e-9
SCORE_TOL = 1e-12


def close(got, want, tol):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    err = float(np.abs(got - want).max()) if want.size else 0.0
    assert err <= tol * scale, f"max |diff| = {err} (scale {scale})"


def plain_rows(ctx, rows_a, cat_a, rows_b, cat_b, wf_idx=None):
    """from_dmxs through the C ABI: two ragged row sets, row r against row r."""
    ea, eb = ctx.envset_from_ragged_rows(rows_a, cat_a), ctx.envset_from_ragged_rows(rows_b, cat_b)
    n = len(rows_a)
    s = ctx.score_pairs(ea, eb, np.stack([np.arange(n)] * 2, axis=1).astype(np.uint32), wf_idx=wf_idx)
    ea.close(); eb.close()
    return s


def plain_coords(ctx, xa, ca, xb, cb, wf_idx=None):
    ea, eb = ctx.envset_from_coords(xa, ca), ctx.envset_from_coords(xb, cb)
    n = len(ca)
    s = ctx.score_pairs(ea, eb, np.stack([np.arange(n)] * 2, axis=1).astype(np.uint32), wf_idx=wf_idx)
    ea.close(); eb.close()
    return s


def case(gpu_ctx, oracle_mod, wf, sd):
    k = sorted(WFS).index(wf) + 4 * sorted(SDS).index(sd)
    cat_w = None if k % 2 == 0 else (0.6, 1.7, 1.1)
    op = set_both(gpu_ctx, oracle_mod, 3, [WFS[wf]], cat_w, SDS[sd])
    weights = np.linspace(-0.7, 1.9, 12) if k % 4 == 1 else None
    return k, op, weights


# --------------------------------------------------------------------------------------- reference parity
@pytest.mark.parametrize("wf", sorted(WFS))
@pytest.mark.parametrize("sd", sorted(SDS))
def test_rows_and_coords_match_the_reference(gpu_ctx, oracle_mod, wf, sd):
    k, op, weights = case(gpu_ctx, oracle_mod, wf, sd)
    xa, ca, xb, cb = rr.tie_free_clouds(400 + k, kinks([WFS[wf]]), n=12)
    ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
    s, ga, gb = gpu_ctx.from_rows_grad(ta, ca, tb, cb, pair_weights=weights)
    rs, ra, rb = rr.from_rows_grad(oracle_mod, op, ta, ca, tb, cb, pair_weights=weights)
    assert np.abs(s - plain_rows(gpu_ctx, ta, ca, tb, cb)).max() <= SCORE_TOL
    assert np.abs(s - rs).max() <= 1e-9
    assert ga.shape == ta.shape and gb.shape == tb.shape
    close(ga, np.array(ra), GRAD_TOL)
    close(gb, np.array(rb), GRAD_TOL)
    cs, cga, cgb = gpu_ctx.from_coords_grad(xa, ca, xb, cb, pair_weights=weights)
    assert np.abs(cs - plain_coords(gpu_ctx, xa, ca, xb, cb)).max() <= SCORE_TOL
    _, wa, wb = rr.from_coords_grad(oracle_mod, op, xa, ca, xb, cb, pair_weights=weights)
    close(cga, wa, GRAD_TOL)
    close(cgb, wb, GRAD_TOL)


def test_per_row_weight_functions_and_pair_weights(gpu_ctx, oracle_mod):
    wfs = [WFS[w] for w in sorted(WFS)]
    op = set_both(gpu_ctx, oracle_mod, 3, wfs, (1.3, 0.4, 0.9), SDS["Kullback-Leibler"])
    xa, ca, xb, cb = rr.tie_free_clouds(7, kinks(wfs), n=12)
    wf_idx = (np.arange(12) % 4).astype(np.uint32)
    weights = np.linspace(-0.7, 1.9, 12)
    weights[5] = 0.0
    ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
    s, ga, gb = gpu_ctx.from_rows_grad(ta, ca, tb, cb, wf_idx=wf_idx, pair_weights=weights)
    assert np.abs(s - plain_rows(gpu_ctx, ta, ca, tb, cb, wf_idx=wf_idx)).max() <= SCORE_TOL
    _, ra, rb = rr.from_rows_grad(oracle_mod, op, ta, ca, tb, cb, wf_idx=wf_idx, pair_weights=weights)
    close(ga, np.array(ra), GRAD_TOL)
    close(gb, np.array(rb), GRAD_TOL)
    assert not ga[5].any() and not gb[5].any()
    _, cga, cgb = gpu_ctx.from_coords_grad(xa, ca, xb, cb, wf_idx=wf_idx, pair_weights=weights)
    _, wa, wb = rr.from_coords_grad(oracle_mod, op, xa, ca, xb, cb, wf_idx=wf_idx, pair_weights=weights)
    close(cga, wa, GRAD_TOL)
    close(cgb, wb, GRAD_TOL)


def test_ragged_rows(gpu_ctx, oracle_mod):
    """Rows of different lengths (the shape of test_ragged_distance_rows, +inf bans included): the gradients come
    back in the ragged layout."""
    op = set_both(gpu_ctx, oracle_mod, 3, [WFS["kumaraswamy"]], (0.6, 1.7, 1.1), SDS["Renyi"])
    ra, ca, rb, cb = rr.tie_free_ragged_rows(99, kinks([WFS["kumaraswamy"]]), n_rows=20, max_len=40)
    ra[3][np.argmax(ra[3])] = np.inf
    weights = np.linspace(-0.7, 1.9, len(ra))
    s, ga, gb = gpu_ctx.from_rows_grad(ra, ca, rb, cb, pair_weights=weights)
    rs, wa, wb = rr.from_rows_grad(oracle_mod, op, ra, ca, rb, cb, pair_weights=weights)
    assert np.abs(s - plain_rows(gpu_ctx, ra, ca, rb, cb)).max() <= SCORE_TOL
    assert isinstance(ga, list) and [len(g) for g in ga] == [len(r) for r in ra] and [len(g) for g in gb] == [len(r) for r in rb]
    close(np.concatenate(ga), np.concatenate(wa), GRAD_TOL)
    close(np.concatenate(gb), np.concatenate(wb), GRAD_TOL)
    assert ga[3][np.argmax(ra[3])] == 0.0


# ------------------------------------------------------------------------------ the ensemble callers' +inf form
def test_ensemble_dmx_form_chains_to_the_cutoff_gradients(gpu_ctx, oracle_mod):
    """compare_ensembles.py's from_dmxs form (+inf at homo-residue entries) and the cutoff form (threshold 10, hetero
    contacts) give the same scores; through the host chain rule over the finite entries, from_rows_grad gives the
    coordinate gradients of from_primitives_grad (uniform [3, 10] has density 0 beyond 10)."""
    base = synth.gen(9, 60, 8, 7)
    a, b = synth.config5_member(base, 0), synth.config5_member(base, 1)
    set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0))], tag_rule={"accept_same": False})
    anchors = np.stack([np.arange(a.n)] * 2, axis=1).astype(np.uint32)
    cs, cga, cgb = gpu_ctx.from_primitives_grad(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0)

    def dmx(c):
        d = rr.euclidean_rows(c.xyz)
        same = c.tag[:, None] == c.tag[None, :]
        np.fill_diagonal(same, False)
        d[same] = np.inf
        return d, same
    (da, ba), (db, bb) = dmx(a), dmx(b)
    s, ga, gb = gpu_ctx.from_rows_grad(da, a.cat, db, b.cat)
    assert np.abs(s - cs).max() <= 1e-12
    assert (ga[ba] == 0.0).all() and (gb[bb] == 0.0).all()
    close(rr.chain_rule(a.xyz, ga), cga, 1e-12)
    close(rr.chain_rule(b.xyz, gb), cgb, 1e-12)


def test_coords_grad_is_rows_grad_and_the_chain_rule(gpu_ctx, oracle_mod):
    set_both(gpu_ctx, oracle_mod, 7, [("dagum", (2.5, 6.0, 1.3))], None, ("Hellinger", (2.0,)))
    a, b = synth.config1()
    n = min(a.n, b.n)
    xa, xb, ca, cb = a.xyz[:n], b.xyz[:n], a.cat[:n], b.cat[:n]
    w = np.random.default_rng(3).normal(size=n)
    s, ga, gb = gpu_ctx.from_coords_grad(xa, ca, xb, cb, pair_weights=w)
    rs, ra, rb = gpu_ctx.from_rows_grad(rr.euclidean_rows(xa), ca, rr.euclidean_rows(xb), cb, pair_weights=w)
    assert np.array_equal(s, rs)
    close(ga, rr.chain_rule(xa, ra), 1e-12)
    close(gb, rr.chain_rule(xb, rb), 1e-12)


def test_repeated_calls_are_byte_identical(gpu_ctx, oracle_mod):
    set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0))])
    a, b = synth.config1()
    n = min(a.n, b.n)
    args = (a.xyz[:n], a.cat[:n], b.xyz[:n], b.cat[:n])
    w = np.random.default_rng(4).normal(size=n)
    first = gpu_ctx.from_coords_grad(*args, pair_weights=w)
    second = gpu_ctx.from_coords_grad(*args, pair_weights=w)
    for x, y in zip(first, second):
        assert x.tobytes() == y.tobytes()
    rows = (rr.euclidean_rows(a.xyz[:n]), a.cat[:n], rr.euclidean_rows(b.xyz[:n]), b.cat[:n])
    first = gpu_ctx.from_rows_grad(*rows, pair_weights=w)
    second = gpu_ctx.from_rows_grad(*rows, pair_weights=w)
    for x, y in zip(first, second):
        assert x.tobytes() == y.tobytes()


def test_large_rows(gpu_ctx, oracle_mod):
    """n = 3000 points: rows far beyond every shared-memory sort class and staging limit.  All scores against
    from_coords; the coordinate gradient of a sample of rows (the other rows weighted 0) against the reference."""
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0))])
    rng = np.random.default_rng(5)
    n = 3000
    xa = rng.uniform(0, 40, (n, 3))
    xb = xa + rng.normal(0, 0.7, (n, 3))
    ca = rng.integers(0, 7, n).astype(np.uint16)
    cb = ca.copy()
    cb[rng.integers(0, n, 300)] = rng.integers(0, 7, 300)
    s, _, _ = gpu_ctx.from_coords_grad(xa, ca, xb, cb)
    assert np.abs(s - plain_coords(gpu_ctx, xa, ca, xb, cb)).max() <= SCORE_TOL
    sample = rng.choice(n, 3, replace=False)
    w = np.zeros(n)
    w[sample] = [1.0, -0.5, 2.0]
    _, ga, gb = gpu_ctx.from_coords_grad(xa, ca, xb, cb, pair_weights=w)
    want = [np.zeros((n, 3)), np.zeros((n, 3))]
    ta, tb = (rr.euclidean_rows(x) for x in (xa, xb))
    for r in sample:
        _, g_a, g_b = rr.row_pair_grad(oracle_mod, op, ta[r], ca, tb[r], cb, 0, w[r])
        for side, (x, t, g) in enumerate(((xa, ta, g_a), (xb, tb, g_b))):
            live = t[r] > 0
            c = np.where(live, g / np.where(live, t[r], 1.0), 0.0)
            d = x[r][None, :] - x
            want[side][r] += (c[:, None] * d).sum(axis=0)
            want[side] -= c[:, None] * d
    close(ga, want[0], GRAD_TOL)
    close(gb, want[1], GRAD_TOL)


@pytest.mark.parametrize("wf", sorted(WFS))
def test_directional_derivative_matches_finite_differences(gpu_ctx, oracle_mod, wf):
    h = 1e-4
    set_both(gpu_ctx, oracle_mod, 3, [WFS[wf]], (0.8, 1.2, 1.0), SDS["Hellinger"])
    xa, ca, xb, cb = rr.tie_free_clouds(500 + sorted(WFS).index(wf), kinks([WFS[wf]]), n=10, gap=100 * h)
    rng = np.random.default_rng(5)
    va, vb = rng.normal(size=xa.shape), rng.normal(size=xb.shape)
    norm = np.sqrt((va ** 2).sum() + (vb ** 2).sum())
    va, vb = va / norm, vb / norm
    _, ga, gb = gpu_ctx.from_coords_grad(xa, ca, xb, cb)
    along = float((ga * va).sum() + (gb * vb).sum())

    def S(t):
        return plain_coords(gpu_ctx, xa + t * va, ca, xb + t * vb, cb).sum()
    fd = (S(h) - S(-h)) / (2 * h)
    gnorm = np.sqrt((ga ** 2).sum() + (gb ** 2).sum())
    assert gnorm > 0
    assert abs(fd - along) <= 1e-5 * gnorm, (fd, along, gnorm)


def test_autograd_function_passes_gradcheck(gpu_ctx, oracle_mod):
    """The torch.autograd.Function of INTEGRATION.md for from_coords: forward = from_coords, backward =
    from_coords_grad with the upstream gradient as pair weights."""
    import torch

    import loco_hd

    names = ["X", "Y", "Z"]
    lchd = loco_hd.LoCoHD(names, loco_hd.WeightFunction("hyper_exp", list(WFS["hyper_exp"][1])))
    xa, ca, xb, cb = rr.tie_free_clouds(71, [], n=8)
    seq_a, seq_b = [names[c] for c in ca], [names[c] for c in cb]

    class LoCoHDCoords(torch.autograd.Function):
        @staticmethod
        def forward(fctx, xyz_a, xyz_b, lchd, seq_a, seq_b):
            fctx.save_for_backward(xyz_a, xyz_b)
            fctx.args = (lchd, seq_a, seq_b)
            s = lchd.from_coords(seq_a, seq_b, xyz_a.detach().cpu().numpy(), xyz_b.detach().cpu().numpy())
            return torch.tensor(s, dtype=xyz_a.dtype, device=xyz_a.device)

        @staticmethod
        def backward(fctx, grad_output):
            xyz_a, xyz_b = fctx.saved_tensors
            lchd, seq_a, seq_b = fctx.args
            _, ga, gb = lchd.from_coords_grad(seq_a, seq_b, xyz_a.detach().cpu().numpy(), xyz_b.detach().cpu().numpy(),
                                              pair_weights=grad_output.detach().cpu().numpy())
            return torch.from_numpy(ga).to(xyz_a.device), torch.from_numpy(gb).to(xyz_b.device), None, None, None

    xa_t = torch.tensor(xa, dtype=torch.float64, device="cuda", requires_grad=True)
    xb_t = torch.tensor(xb, dtype=torch.float64, device="cuda", requires_grad=True)
    assert torch.autograd.gradcheck(lambda a, b: LoCoHDCoords.apply(a, b, lchd, seq_a, seq_b), (xa_t, xb_t), eps=1e-6,
                                    atol=1e-6, rtol=1e-4)


def test_device_inputs_and_outputs(gpu_ctx, oracle_mod):
    """Inputs and outputs as torch CUDA tensors (raw pointers): the same bytes as numpy arrays."""
    import torch

    set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0)), ("dagum", (2.5, 6.0, 1.3))])
    a, b = synth.config1()
    n = min(a.n, b.n)
    xa, xb, ca, cb = a.xyz[:n], b.xyz[:n], a.cat[:n], b.cat[:n]
    rng = np.random.default_rng(19)
    wf_idx = rng.integers(0, 2, n).astype(np.uint32)
    w = rng.normal(size=n)
    hs, ha, hb = gpu_ctx.from_coords_grad(xa, ca, xb, cb, wf_idx=wf_idx, pair_weights=w)
    dev = [torch.from_numpy(np.ascontiguousarray(x)).cuda()
           for x in (xa, ca.view(np.int16), xb, cb.view(np.int16), wf_idx.view(np.int32), w)]
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    oa = torch.full((n, 3), 7.0, dtype=torch.float64, device="cuda")
    ob = torch.full((n, 3), 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    p = [t.data_ptr() for t in dev]
    gpu_ctx.from_coords_grad(p[0], p[1], p[2], p[3], wf_idx=p[4], pair_weights=p[5], out=out.data_ptr(),
                             grad_a=oa.data_ptr(), grad_b=ob.data_ptr(), n_points=n)
    torch.cuda.synchronize()
    assert out.cpu().numpy().tobytes() == hs.tobytes()
    assert oa.cpu().numpy().tobytes() == ha.tobytes() and ob.cpu().numpy().tobytes() == hb.tobytes()
    # rows: device values, weights and outputs (offsets and categories on the host)
    ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
    rs, ra, rb = gpu_ctx.from_rows_grad(ta, ca, tb, cb, wf_idx=wf_idx, pair_weights=w)
    offs = (np.arange(n + 1) * n).astype(np.uint64)
    dv = [torch.from_numpy(t.ravel()).cuda() for t in (ta, tb)]
    ra_d = torch.empty(n * n, dtype=torch.float64, device="cuda")
    rb_d = torch.empty(n * n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    gpu_ctx.from_rows_grad(dv[0].data_ptr(), ca, dv[1].data_ptr(), cb, wf_idx=p[4], pair_weights=p[5],
                           out=out.data_ptr(), grad_a=ra_d.data_ptr(), grad_b=rb_d.data_ptr(), offsets_a=offs,
                           offsets_b=offs)
    torch.cuda.synchronize()
    assert out.cpu().numpy().tobytes() == rs.tobytes()
    assert ra_d.cpu().numpy().tobytes() == ra.tobytes() and rb_d.cpu().numpy().tobytes() == rb.tobytes()


# ------------------------------------------------------------------------------------------------------ errors
def test_errors_match_from_dmxs_and_from_coords(gpu_ctx, oracle_mod):
    from loco_hd_b200._capi import LocoHDError

    set_both(gpu_ctx, oracle_mod, 3, [WFS["uniform"]], None, SDS["Hellinger"])
    xa, ca, xb, cb = rr.tie_free_clouds(41, [], n=8)
    ta, tb = rr.euclidean_rows(xa), rr.euclidean_rows(xb)
    no_zero = ta.copy()
    no_zero[2, 2] = 0.5
    bad_cat = ca.copy()
    bad_cat[4] = 9
    nan_xyz = xa.copy()
    nan_xyz[3, 1] = np.nan
    rows_cases = [([list(r) for r in ta], ca[:5], [list(r) for r in tb], cb),   # short category list
                  ([list(r) for r in ta[:3]] + [[]] + [list(r) for r in ta[4:]], ca, [list(r) for r in tb], cb),
                  (no_zero, ca, tb, cb), (ta, bad_cat, tb, cb)]
    for A, cA, B, cB in rows_cases:
        with pytest.raises(LocoHDError) as plain:
            plain_rows(gpu_ctx, A, cA, B, cB)
        with pytest.raises(LocoHDError) as grad:
            gpu_ctx.from_rows_grad(A, cA, B, cB)
        assert grad.value.status == plain.value.status and str(grad.value) == str(plain.value)
    for X, cX in ((nan_xyz, ca), (xa, bad_cat)):
        with pytest.raises(LocoHDError) as plain:
            plain_coords(gpu_ctx, X, cX, xb, cb)
        with pytest.raises(LocoHDError) as grad:
            gpu_ctx.from_coords_grad(X, cX, xb, cb)
        assert grad.value.status == plain.value.status and str(grad.value) == str(plain.value)
    with pytest.raises(LocoHDError) as grad:
        gpu_ctx.from_coords_grad(xa, ca, xb, cb, wf_idx=np.full(8, 3, np.uint32))
    assert grad.value.status == 10
    gpu_ctx.from_coords_grad(xa, ca, xb, cb)   # the context is usable afterwards


def test_python_api_errors_match(gpu_ctx, oracle_mod):
    import loco_hd

    names = ["X", "Y", "Z"]
    one = loco_hd.LoCoHD(names, loco_hd.WeightFunction("uniform", [3.0, 10.0]))
    many = loco_hd.LoCoHD(names, {"u": loco_hd.WeightFunction("uniform", [3.0, 10.0]),
                                  "d": loco_hd.WeightFunction("dagum", [2.5, 6.0, 1.3])})
    xa, ca, xb, cb = rr.tie_free_clouds(43, [], n=6)
    sa, sb = [names[c] for c in ca], [names[c] for c in cb]
    ta, tb = rr.euclidean_rows(xa).tolist(), rr.euclidean_rows(xb).tolist()
    nan_xyz = xa.copy()
    nan_xyz[1, 1] = np.nan
    dmx_cases = [(one, (sa, sb, ta, tb[:-1]), {}),                       # length mismatch
                 (one, (sa[:3], sb, ta, tb), {}),                       # short category list
                 (one, (sa, sb, ta[:2] + [[]] + ta[3:], tb), {}),       # empty row
                 (one, (sa, sb, [[0.5] + r[1:] for r in ta], tb), {}),  # row without a zero
                 (one, (["Q"] + sa[1:], sb, ta, tb), {}),               # unknown category
                 (many, (sa, sb, ta, tb), {"w_func_keys": ["u", "x", "d", "u", "u", "u"]})]   # unknown key
    for lchd, args, kw in dmx_cases:
        with pytest.raises(Exception) as plain:
            lchd.from_dmxs(*args, **kw)
        with pytest.raises(Exception) as grad:
            lchd.from_dmxs_grad(*args, **kw)
        assert type(grad.value) is type(plain.value) and str(grad.value) == str(plain.value)
    coord_cases = [(one, (sa, sb, xa, xb[:-1]), {}), (one, (sa, sb, nan_xyz, xb), {}),
                   (one, (["Q"] + sa[1:], sb, xa, xb), {}),
                   (many, (sa, sb, xa, xb), {"w_func_keys": ["u", "x", "d", "u", "u", "u"]})]
    for lchd, args, kw in coord_cases:
        with pytest.raises(Exception) as plain:
            lchd.from_coords(*args, **kw)
        with pytest.raises(Exception) as grad:
            lchd.from_coords_grad(*args, **kw)
        assert type(grad.value) is type(plain.value) and str(grad.value) == str(plain.value)


# -------------------------------------------------------------------------------------------------- Python API
def test_python_api_matches_the_c_abi(gpu_ctx, oracle_mod):
    import loco_hd

    names = ["X", "Y", "Z"]
    lchd = loco_hd.LoCoHD(names, {"k": loco_hd.WeightFunction("kumaraswamy", list(WFS["kumaraswamy"][1])),
                                  "u": loco_hd.WeightFunction("uniform", list(WFS["uniform"][1]))},
                          statistical_distance=loco_hd.StatisticalDistance("Renyi", [1.7, 0.2]))
    set_both(gpu_ctx, oracle_mod, 3, [WFS["kumaraswamy"], WFS["uniform"]], None, SDS["Renyi"])
    xa, ca, xb, cb = rr.tie_free_clouds(61, kinks([WFS["kumaraswamy"], WFS["uniform"]]), n=10)
    sa, sb = [names[c] for c in ca], [names[c] for c in cb]
    keys = ["k", "u"] * 5
    wf_idx = np.array([0, 1] * 5, np.uint32)   # the keys in sorted order: "k" = 0, "u" = 1
    w = np.linspace(0.5, 1.5, 10)
    s, ga, gb = lchd.from_coords_grad(sa, sb, xa.tolist(), xb.tolist(), w_func_keys=keys, pair_weights=w)
    cs, ca_, cb_ = gpu_ctx.from_coords_grad(xa, ca, xb, cb, wf_idx=wf_idx, pair_weights=w)
    assert np.array_equal(s, cs) and np.array_equal(ga, ca_) and np.array_equal(gb, cb_)
    assert np.abs(s - np.array(lchd.from_coords(sa, sb, xa, xb, w_func_keys=keys))).max() <= SCORE_TOL
    ta, tb = rr.euclidean_rows(xa).tolist(), rr.euclidean_rows(xb).tolist()
    s, ga, gb = lchd.from_dmxs_grad(sa, sb, ta, tb, w_func_keys=keys, pair_weights=w)
    cs, ra, rb = gpu_ctx.from_rows_grad(np.array(ta), ca, np.array(tb), cb, wf_idx=wf_idx, pair_weights=w)
    assert np.array_equal(s, cs) and np.array_equal(ga, ra) and np.array_equal(gb, rb)
    assert ga.shape == (10, 10)
    ragged_a = [r[:max(i + 1, 6 + i % 4)] for i, r in enumerate(ta)]   # row i keeps its zero at column i
    s, ga, gb = lchd.from_dmxs_grad(sa, sb, ragged_a, tb, w_func_keys=keys)
    cs, ra, rb = gpu_ctx.from_rows_grad(ragged_a, ca, tb, cb, wf_idx=wf_idx)
    assert np.array_equal(s, cs)
    assert isinstance(ga, list) and all(np.array_equal(x, y) for x, y in zip(ga, ra))
    assert np.abs(s - np.array(lchd.from_dmxs(sa, sb, ragged_a, tb, w_func_keys=keys))).max() <= SCORE_TOL
    with pytest.raises(ValueError):
        lchd.from_coords_grad(sa, sb, xa, xb, w_func_keys=keys, pair_weights=w[:-1])
