"""GPU tests of the coordinate gradients of LoCoHD scores (locohd_from_primitives_grad, LoCoHD.from_arrays_grad).

Scores must equal those of from_primitives (1e-12) and of the oracle (1e-9); gradients must equal those of the CPU
reference in tests/grad_reference.py (1e-9 relative to max(1, max |g|)), whose own gradients are checked against
finite differences of the oracle in tests/test_grad_oracle.py.  Every gather route and upload route must give the
same gradients (1e-12), and directional derivatives must match finite differences of the existing from_primitives.
"""
import numpy as np
import pytest

import grad_reference as gr
from benchdata import synth
from grad_reference import SDS, THRESHOLD, WFS, tie_free_case
from helpers import assert_scores_close, set_both

pytestmark = pytest.mark.gpu

GRAD_TOL = 1e-9
ROUTE_TOL = 1e-12


def close(got, want, tol):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    err = float(np.abs(got - want).max()) if want.size else 0.0
    assert err <= tol * scale, f"max |diff| = {err} (scale {scale})"


def grad_call(ctx, A, B, anchors, threshold, **kw):
    return ctx.from_primitives_grad(*A, *B, np.asarray(anchors, np.uint32).reshape(-1, 2), threshold, **kw)


def check_against_reference(ctx, oracle_mod, op, A, B, anchors, threshold, wf_idx=None, pair_weights=None):
    s, ga, gb = grad_call(ctx, A, B, anchors, threshold, wf_idx=wf_idx, pair_weights=pair_weights)
    plain = ctx.from_primitives(*A, *B, np.asarray(anchors, np.uint32).reshape(-1, 2), threshold, wf_idx=wf_idx)
    assert np.abs(s - plain).max() <= 1e-12
    rs, ra, rb = gr.from_primitives_grad(oracle_mod, op, *A, *B, anchors, threshold,
                                         wf_idx=None if wf_idx is None else np.asarray(wf_idx),
                                         pair_weights=pair_weights)
    assert_scores_close(s, oracle_mod.from_primitives(op, *A, *B, anchors, threshold, wf_idx=wf_idx))
    close(ga, ra, GRAD_TOL)
    close(gb, rb, GRAD_TOL)
    return s, ga, gb


# ------------------------------------------------------------------------------------ 1, 2: scores and gradients
@pytest.mark.parametrize("wf", sorted(WFS))
@pytest.mark.parametrize("sd", sorted(SDS))
def test_gradients_match_the_reference(gpu_ctx, oracle_mod, wf, sd):
    """The cases of the CPU file: every weight-function family x every statistical distance, with category weights,
    both tag-rule kinds and pair weights varying with the case."""
    k = sorted(WFS).index(wf) + 4 * sorted(SDS).index(sd)
    cat_w = None if k % 2 == 0 else (0.6, 1.7, 1.1)
    tag_rule = [{"accept_same": True}, {"accept_same": False},
                {"tag_pairs": [(0, 1), (1, 2)], "accepted_pairs": True, "ordered": False}][k % 3]
    op = set_both(gpu_ctx, oracle_mod, 3, [WFS[wf]], cat_w, SDS[sd], tag_rule)
    A, B, anchors = tie_free_case(100 + k, [WFS[wf]])
    weights = np.linspace(-0.7, 1.9, len(anchors)) if k % 4 == 1 else None
    check_against_reference(gpu_ctx, oracle_mod, op, A, B, anchors, THRESHOLD, pair_weights=weights)


def test_gradients_per_pair_weight_functions(gpu_ctx, oracle_mod):
    wfs = [WFS[w] for w in sorted(WFS)]
    op = set_both(gpu_ctx, oracle_mod, 3, wfs, (1.3, 0.4, 0.9), SDS["Kullback-Leibler"],
                  {"tag_pairs": [(0, 0), (2, 1)], "accepted_pairs": False, "ordered": True})
    A, B, anchors = tie_free_case(7, wfs)
    wf_idx = (np.arange(len(anchors)) % 4).astype(np.uint32)
    check_against_reference(gpu_ctx, oracle_mod, op, A, B, anchors, THRESHOLD, wf_idx=wf_idx,
                            pair_weights=np.linspace(-0.7, 1.9, len(anchors)))


def test_config2_shaped_pair(gpu_ctx, oracle_mod):
    """A configuration-2-shaped pair (10 000 primitives, 10 000 anchor pairs): all scores against from_primitives,
    and scores and gradients of a sample of 24 anchor pairs against the reference."""
    a, b = synth.config2_pair(0)
    A, B = (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag)
    op = set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0))], tag_rule={"accept_same": False})
    anchors = np.stack([np.arange(a.n), np.arange(b.n)], axis=1).astype(np.uint32)
    s, ga, gb = grad_call(gpu_ctx, A, B, anchors, 10.0)
    assert np.abs(s - gpu_ctx.from_primitives(*A, *B, anchors, 10.0)).max() <= 1e-12
    assert np.isfinite(ga).all() and np.isfinite(gb).all() and np.abs(ga).max() > 0
    sample = anchors[np.random.default_rng(3).choice(len(anchors), 24, replace=False)]
    check_against_reference(gpu_ctx, oracle_mod, op, A, B, sample, 10.0)


# ------------------------------------------------------------------------------ 3: finite differences of the GPU
@pytest.mark.parametrize("wf", sorted(WFS))
def test_directional_derivative_matches_finite_differences(gpu_ctx, oracle_mod, wf):
    h = 1e-4
    set_both(gpu_ctx, oracle_mod, 3, [WFS[wf]], (0.8, 1.2, 1.0), SDS["Hellinger"], {"accept_same": False})
    A, B, anchors = tie_free_case(300 + sorted(WFS).index(wf), [WFS[wf]], n=10, gap=100 * h)
    rng = np.random.default_rng(5)
    va, vb = rng.normal(size=A[0].shape), rng.normal(size=B[0].shape)
    norm = np.sqrt((va ** 2).sum() + (vb ** 2).sum())
    va, vb = va / norm, vb / norm
    _, ga, gb = grad_call(gpu_ctx, A, B, anchors, THRESHOLD)
    along = float((ga * va).sum() + (gb * vb).sum())

    def S(t):
        return gpu_ctx.from_primitives(A[0] + t * va, A[1], A[2], B[0] + t * vb, B[1], B[2], anchors, THRESHOLD).sum()
    fd = (S(h) - S(-h)) / (2 * h)
    gnorm = np.sqrt((ga ** 2).sum() + (gb ** 2).sum())
    assert gnorm > 0
    assert abs(fd - along) <= 1e-5 * gnorm, (fd, along, gnorm)


# ----------------------------------------------------------------------------------------------- leaf math: w(x)
DENSITY_WFS = [("hyper_exp", (1.0, 2.0, 0.5, 0.15)), ("hyper_exp", (1.0, 1.0)),
               ("dagum", (2.5, 3.0, 1.3)), ("dagum", (0.5, 3.0, 1.0)), ("dagum", (1.0, 3.0, 1.0)),
               ("uniform", (1.5, 5.0)), ("uniform", (3.0, 10.0)),
               ("kumaraswamy", (3.0, 10.0, 2.0, 5.0)), ("kumaraswamy", (5.0, 9.0, 7.0, 7.0)),
               ("kumaraswamy", (0.0, 3.0, 1.0, 3.0)), ("kumaraswamy", (1.0, 5.5, 2.3, 1.7))]


@pytest.mark.parametrize("name,params", DENSITY_WFS)
def test_weight_function_densities(gpu_ctx, name, params):
    """locohd_wf_density_points on the device against the reference density and against a numerical derivative of
    the device CDF (locohd_wf_integral_points): all four families, integer (powi_small) and non-integer kumaraswamy
    exponents, dagum at 0 and tiny x, points exactly at and on both sides of x_min / x_max."""
    x = [0.05, 0.7, 1.6, 2.2, 3.7, 4.1, 5.4, 6.3, 7.0, 8.8, 11.0, 30.0]
    kinks = list(params[:2]) if name in ("uniform", "kumaraswamy") else []
    for k in kinks:
        x += [k, np.nextafter(k, -np.inf), np.nextafter(k, np.inf), k - 1e-4, k + 1e-4]
    if name == "dagum":
        x += [0.0, 5e-324, 1e-308, 1e-300, 1e-6, 1e-3]
    x = np.array(sorted(v for v in x if v >= 0.0))
    got = gpu_ctx.wf_density_points(name, params, x)
    ref = np.array([gr.wf_density(name, params, float(v)) for v in x])
    assert not np.isnan(got).any()
    assert np.array_equal(np.isinf(got), np.isinf(ref)), (x, got, ref)
    fin = np.isfinite(ref)
    err = np.abs(got[fin] - ref[fin]) / np.maximum(1.0, np.abs(ref[fin]))
    # 1e-10: at x_max a non-integer exponent b < 2 turns the one-ulp difference of the CDF's z = (x - x_min) / range
    # (computed as a product with 1 / range, as in the CDF) into ~1e-11 of (1 - z^a)^(b - 1)
    assert err.max() <= 1e-10, (x[fin][err.argmax()], got[fin][err.argmax()], ref[fin][err.argmax()])
    # numerical derivative of the device CDF away from the kinks
    far = np.array([v >= 1e-300 and all(abs(v - k) > 1e-3 for k in kinks) for v in x])   # x / 4 representable
    h = np.minimum(1e-6, x[far] * 1e-4)   # relative steps: dagum with a p < 1 is singular at 0
    cdf = gpu_ctx.wf_integral_points(name, params, np.concatenate([x[far] + h, x[far] - h]))
    num = (cdf[:far.sum()] - cdf[far.sum():]) / (2 * h)
    assert np.all(np.abs(got[far] - num) <= 1e-6 * np.maximum(1.0, np.abs(num))), (x[far], got[far], num)


def test_gradients_integer_kumaraswamy(gpu_ctx, oracle_mod):
    """The reference API's own Kumaraswamy (3, 10, 2, 5): integer exponents, so the device takes powi_small."""
    wf = ("kumaraswamy", (3.0, 10.0, 2.0, 5.0))
    op = set_both(gpu_ctx, oracle_mod, 3, [wf], (0.6, 1.7, 1.1), SDS["Hellinger"], {"accept_same": False})
    A, B, anchors = tie_free_case(81, [wf])
    check_against_reference(gpu_ctx, oracle_mod, op, A, B, anchors, THRESHOLD,
                            pair_weights=np.linspace(-0.7, 1.9, len(anchors)))


# ------------------------------------------------------------------------------------------------ 4: pair weights
def test_pair_weights(gpu_ctx, oracle_mod):
    import torch

    set_both(gpu_ctx, oracle_mod, 3, [WFS["kumaraswamy"]], None, SDS["Hellinger"])
    A, B, anchors = tie_free_case(11, [WFS["kumaraswamy"]])
    w = np.array([0.3, -1.2, 2.5, 0.0, 0.9])[:len(anchors)]
    s, ga, gb = grad_call(gpu_ctx, A, B, anchors, THRESHOLD, pair_weights=w)
    sum_a, sum_b = np.zeros_like(ga), np.zeros_like(gb)
    for p in range(len(anchors)):
        sp, pa, pb = grad_call(gpu_ctx, A, B, anchors[p:p + 1], THRESHOLD)
        assert sp[0] == s[p]
        sum_a += w[p] * pa
        sum_b += w[p] * pb
    close(ga, sum_a, ROUTE_TOL)
    close(gb, sum_b, ROUTE_TOL)
    s0, za, zb = grad_call(gpu_ctx, A, B, anchors, THRESHOLD, pair_weights=np.zeros(len(anchors)))
    assert np.array_equal(s0, s) and not za.any() and not zb.any()
    dw = torch.from_numpy(w).cuda()
    torch.cuda.synchronize()
    sd, da, db = grad_call(gpu_ctx, A, B, anchors, THRESHOLD, pair_weights=dw.data_ptr())
    assert np.array_equal(sd, s)
    close(da, ga, ROUTE_TOL)
    close(db, gb, ROUTE_TOL)


# ------------------------------------------------------------------------------------------------ 5: gather routes
def dense_pair(seed, n, extent):
    rng = np.random.default_rng(seed)
    A = (rng.uniform(-extent, extent, (n, 3)), rng.integers(0, 5, n).astype(np.uint16), np.zeros(n, np.uint32))
    B = (A[0] + rng.normal(0, 0.5, (n, 3)), A[1].copy(), A[2].copy())
    centre = np.flatnonzero(np.abs(A[0]).max(axis=1) < extent / 4)[:40]
    return A, B, np.stack([centre, centre], axis=1).astype(np.uint32)


@pytest.mark.parametrize("members", [700, 1500])
def test_large_environments_and_the_multi_kernel_gather(gpu_ctx, oracle_mod, monkeypatch, members):
    """Environments above 512 members (the fused 1024-member gather) and above 1024 (the fused gather gives up and the
    multi-kernel gather builds them): scores and gradients of a sample of pairs against the reference.  With
    LOCOHD_LEGACY_GATHER=1 (the multi-kernel gather for every size) the whole call gives the same gradients as the
    default route; at 1500 members both routes are the multi-kernel gather, so there the reference is the check."""
    op = set_both(gpu_ctx, oracle_mod, 5, [("hyper_exp", (1.0, 0.3))], (1.0, 2.0, 0.5, 1.5, 1.0), ("Renyi", (0.6, 0.1)))
    n = 6000
    extent = 0.5 * (n * 4.19 * 6.0 ** 3 / members) ** (1 / 3)   # members within 6 A of a central anchor
    A, B, anchors = dense_pair(members, n, extent)
    env = gpu_ctx.envset_build(gpu_ctx.structure(*A), anchors[:, 0], 6.0, keep_indices=True)
    sizes = np.diff(env.dump()[0])
    assert sizes.max() > (512 if members < 1024 else 1024)
    s, ga, gb = grad_call(gpu_ctx, A, B, anchors, 6.0)
    assert np.abs(s - gpu_ctx.from_primitives(*A, *B, anchors, 6.0)).max() <= 1e-12
    big = np.argsort(sizes)[-3:]   # the largest environments of the call
    check_against_reference(gpu_ctx, oracle_mod, op, A, B, anchors[big], 6.0)
    monkeypatch.setenv("LOCOHD_LEGACY_GATHER", "1")
    sl, la, lb = grad_call(gpu_ctx, A, B, anchors, 6.0)
    assert np.abs(sl - s).max() <= ROUTE_TOL
    close(la, ga, ROUTE_TOL)
    close(lb, gb, ROUTE_TOL)


def test_above_the_staging_limit(gpu_ctx, oracle_mod):
    """A host call whose upload exceeds the 8 MB staging buffer: 200 anchor pairs repeated 3 000 times with weights
    1 / 3 000 give the gradients of the 200 pairs, and the same scores."""
    a = synth.gen(41, 125, 8, 7)
    b = synth.partner(a, 1.0, 42)
    A, B = (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag)
    set_both(gpu_ctx, oracle_mod, 7, [("kumaraswamy", (3.0, 10.0, 2.0, 5.0))], tag_rule={"accept_same": False})
    base = np.random.default_rng(43).integers(0, a.n, size=(200, 2)).astype(np.uint32)
    reps = 3000
    s, ga, gb = grad_call(gpu_ctx, A, B, base, 10.0)
    sw, wa, wb = grad_call(gpu_ctx, A, B, np.tile(base, (reps, 1)), 10.0, pair_weights=np.full(200 * reps, 1 / reps))
    assert np.abs(sw - np.tile(s, reps)).max() <= 1e-12
    close(wa, ga, ROUTE_TOL)
    close(wb, gb, ROUTE_TOL)


def test_device_inputs_and_outputs(gpu_ctx, oracle_mod):
    """Every input and output a torch CUDA tensor (raw pointers): the same scores and gradients as numpy arrays."""
    import torch

    a, b = synth.config1()
    set_both(gpu_ctx, oracle_mod, 7, [("uniform", (3.0, 10.0)), ("dagum", (2.5, 6.0, 1.3))],
             tag_rule={"accept_same": False})
    rng = np.random.default_rng(19)
    anchors = np.stack([rng.permutation(a.n)[:200], rng.permutation(b.n)[:200]], axis=1).astype(np.uint32)
    wf_idx = rng.integers(0, 2, len(anchors)).astype(np.uint32)
    weights = rng.normal(size=len(anchors))
    hs, ha, hb = gpu_ctx.from_primitives_grad(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0,
                                              wf_idx=wf_idx, pair_weights=weights)
    arrays = (a.xyz, a.cat.view(np.int16), a.tag.view(np.int32), b.xyz, b.cat.view(np.int16), b.tag.view(np.int32),
              anchors.view(np.int32), wf_idx.view(np.int32), weights)
    dev = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in arrays]
    out = torch.empty(len(anchors), dtype=torch.float64, device="cuda")
    oa = torch.full((a.n, 3), 7.0, dtype=torch.float64, device="cuda")
    ob = torch.full((b.n, 3), 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ptr = [t.data_ptr() for t in dev]
    gpu_ctx.from_primitives_grad(*ptr[:7], 10.0, wf_idx=ptr[7], pair_weights=ptr[8], out=out.data_ptr(),
                                 grad_a=oa.data_ptr(), grad_b=ob.data_ptr(), n_a=a.n, n_b=b.n, n_pairs=len(anchors))
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), hs)
    close(oa.cpu().numpy(), ha, ROUTE_TOL)
    close(ob.cpu().numpy(), hb, ROUTE_TOL)


# -------------------------------------------------------------------------------------------------- 6: edge cases
def test_primitive_on_top_of_its_anchor(gpu_ctx, oracle_mod):
    set_both(gpu_ctx, oracle_mod, 3, [WFS["dagum"]], None, SDS["Hellinger"])
    A, B, anchors = tie_free_case(21, [WFS["dagum"]])
    B[0][1] = B[0][anchors[0, 1]]
    s, ga, gb = grad_call(gpu_ctx, A, B, anchors, THRESHOLD)
    assert np.isfinite(s).all() and np.isfinite(ga).all() and np.isfinite(gb).all()


def test_renyi_zero_on_disjoint_compositions(gpu_ctx, oracle_mod):
    op = set_both(gpu_ctx, oracle_mod, 2, [("uniform", (0.0, 5.0))], None, ("Renyi", (0.0, 0.0)))
    A, B, anchors = tie_free_case(31, [("uniform", (0.0, 5.0))], C=1)
    B = (B[0], np.ones_like(B[1]), B[2])   # A holds category 0 only, B category 1 only
    s, ga, gb = grad_call(gpu_ctx, A, B, anchors, THRESHOLD)
    rs, ra, rb = gr.from_primitives_grad(oracle_mod, op, *A, *B, anchors, THRESHOLD)
    assert not np.isfinite(rs).all()
    for got, want in ((s, rs), (ga, ra), (gb, rb)):
        assert np.array_equal(np.isfinite(got), np.isfinite(want))
        fin = np.isfinite(want)
        if fin.any():
            close(got[fin], want[fin], GRAD_TOL)


def test_errors_match_from_primitives(gpu_ctx, oracle_mod):
    from loco_hd_b200._capi import LocoHDError

    set_both(gpu_ctx, oracle_mod, 3, [WFS["uniform"]], None, SDS["Hellinger"])
    A, B, anchors = tie_free_case(41, [WFS["uniform"]])
    bad_cat = (A[0], A[1].copy(), A[2])
    bad_cat[1][0] = 9
    nan_xyz = (A[0].copy(), A[1], A[2])
    nan_xyz[0][2, 1] = np.nan
    bad_anchor = anchors.copy()
    bad_anchor[1, 0] = len(A[0])
    for args, thr in (((bad_cat, B, anchors), THRESHOLD), ((nan_xyz, B, anchors), THRESHOLD),
                      ((A, B, bad_anchor), THRESHOLD), ((A, B, anchors), 0.0), ((A, B, anchors), -1.0)):
        X, Y, an = args
        with pytest.raises(LocoHDError) as plain:
            gpu_ctx.from_primitives(*X, *Y, an, thr)
        with pytest.raises(LocoHDError) as grad:
            grad_call(gpu_ctx, X, Y, an, thr)
        assert isinstance(grad.value, ValueError) and grad.value.status == plain.value.status
    # the context is usable afterwards
    grad_call(gpu_ctx, A, B, anchors, THRESHOLD)


def test_no_pairs_leaves_zero_gradients(gpu_ctx, oracle_mod):
    set_both(gpu_ctx, oracle_mod, 3, [WFS["uniform"]], None, SDS["Hellinger"])
    A, B, _ = tie_free_case(51, [WFS["uniform"]])
    ga, gb = np.full((len(A[0]), 3), 7.0), np.full((len(B[0]), 3), 7.0)
    s, ga2, gb2 = gpu_ctx.from_primitives_grad(*A, *B, np.zeros((0, 2), np.uint32), THRESHOLD, grad_a=ga, grad_b=gb)
    assert len(s) == 0 and not ga.any() and not gb.any() and ga2 is ga and gb2 is gb


# ------------------------------------------------------------------------------------------------- 7: Python API
def test_from_arrays_grad_matches_the_c_abi(gpu_ctx, oracle_mod):
    import loco_hd

    lchd = loco_hd.LoCoHD(["X", "Y", "Z"], loco_hd.WeightFunction("kumaraswamy", list(WFS["kumaraswamy"][1])),
                          loco_hd.TagPairingRule({"accept_same": False}))
    set_both(gpu_ctx, oracle_mod, 3, [WFS["kumaraswamy"]], None, ("Hellinger", (2.0,)), {"accept_same": False})
    A, B, anchors = tie_free_case(61, [WFS["kumaraswamy"]])
    weights = np.linspace(0.5, 1.5, len(anchors))
    s, ga, gb = lchd.from_arrays_grad(*A, *B, anchors, THRESHOLD, pair_weights=weights)
    cs, ca, cb = grad_call(gpu_ctx, A, B, anchors, THRESHOLD, pair_weights=weights)
    assert np.array_equal(s, cs)
    assert np.abs(s - lchd.from_arrays(*A, *B, anchors, THRESHOLD)).max() <= 1e-12   # W from exact distances there
    close(ga, ca, ROUTE_TOL)
    close(gb, cb, ROUTE_TOL)
    assert ga.shape == (len(A[0]), 3) and gb.shape == (len(B[0]), 3)
    with pytest.raises(ValueError):
        lchd.from_arrays_grad(*A, *B, anchors, THRESHOLD, pair_weights=weights[:-1])


def test_autograd_function_passes_gradcheck(gpu_ctx, oracle_mod):
    """The torch.autograd.Function of INTEGRATION.md: forward = from_primitives, backward = from_primitives_grad with
    the upstream gradient as pair weights (environments are rebuilt in backward)."""
    import torch

    set_both(gpu_ctx, oracle_mod, 3, [WFS["hyper_exp"]], None, SDS["Hellinger"])
    A, B, anchors = tie_free_case(71, [WFS["hyper_exp"]], n=8)

    class LoCoHDScore(torch.autograd.Function):
        @staticmethod
        def forward(fctx, xyz_a, xyz_b):
            fctx.save_for_backward(xyz_a, xyz_b)
            out = torch.empty(len(anchors), dtype=torch.float64, device=xyz_a.device)
            torch.cuda.synchronize()
            gpu_ctx.from_primitives(xyz_a.data_ptr(), A[1], A[2], xyz_b.data_ptr(), B[1], B[2], anchors, THRESHOLD,
                                    out=out.data_ptr(), n_a=len(A[1]), n_b=len(B[1]), n_pairs=len(anchors))
            return out

        @staticmethod
        def backward(fctx, grad_out):
            xyz_a, xyz_b = fctx.saved_tensors
            grad_out = grad_out.contiguous()
            ga, gb = torch.empty_like(xyz_a), torch.empty_like(xyz_b)
            torch.cuda.synchronize()
            gpu_ctx.from_primitives_grad(xyz_a.data_ptr(), A[1], A[2], xyz_b.data_ptr(), B[1], B[2], anchors,
                                         THRESHOLD, pair_weights=grad_out.data_ptr(), grad_a=ga.data_ptr(),
                                         grad_b=gb.data_ptr(), n_a=len(A[1]), n_b=len(B[1]), n_pairs=len(anchors))
            return ga, gb

    xa = torch.tensor(A[0], dtype=torch.float64, device="cuda", requires_grad=True)
    xb = torch.tensor(B[0], dtype=torch.float64, device="cuda", requires_grad=True)
    assert torch.autograd.gradcheck(LoCoHDScore.apply, (xa, xb), eps=1e-6, atol=1e-6, rtol=1e-4)
