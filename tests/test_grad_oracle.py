"""CPU checks of the gradient reference (tests/grad_reference.py) that the GPU's locohd_from_primitives_grad is
compared with: its weight-function densities against numerical derivatives of the oracle's CDF, and its coordinate
gradients against central finite differences of the oracle's scores."""
import numpy as np
import pytest

import grad_reference as gr
from grad_reference import H, SDS, THRESHOLD, WFS, tie_free_case


def finite_difference(oracle, op, A, B, anchors, wf_idx, weights):
    def f(xa, xb):
        s = oracle.from_primitives(op, xa, A[1], A[2], xb, B[1], B[2], anchors, THRESHOLD, wf_idx=wf_idx)
        return float(np.dot(weights, s))
    grads = []
    for side in (0, 1):
        g = np.zeros((len(A[0]) if side == 0 else len(B[0]), 3))
        for i in range(g.shape[0]):
            for k in range(3):
                xs = [A[0].copy(), B[0].copy()]
                xs[side][i, k] += H
                fp = f(*xs)
                xs[side][i, k] -= 2 * H
                fm = f(*xs)
                g[i, k] = (fp - fm) / (2 * H)
        grads.append(g)
    return grads


def run_case(oracle_mod, wfs, sd, cat_w, tag_rule, seed, per_pair_wf=False, weighted=False):
    op = oracle_mod.Params(3, [list(w) for w in wfs], cat_w, sd, tag_rule)
    A, B, anchors = tie_free_case(seed, wfs)
    P = len(anchors)
    wf_idx = (np.arange(P) % len(wfs)).astype(np.int32) if per_pair_wf else None
    weights = np.linspace(-0.7, 1.9, P) if weighted else np.ones(P)
    s, ga, gb = gr.from_primitives_grad(oracle_mod, op, *A, *B, anchors, THRESHOLD, wf_idx=wf_idx,
                                        pair_weights=weights if weighted else None)
    ref = oracle_mod.from_primitives(op, *A, *B, anchors, THRESHOLD, wf_idx=wf_idx)
    assert np.abs(s - ref).max() <= 1e-12
    fa, fb = finite_difference(oracle_mod, op, A, B, anchors, wf_idx, weights)
    scale = max(np.abs(fa).max(), np.abs(fb).max())
    assert scale > 0
    err = max(np.abs(ga - fa).max(), np.abs(gb - fb).max())
    assert err <= 1e-6 * scale, f"gradient vs finite differences: {err} (max |g| {scale})"


@pytest.mark.parametrize("wf", sorted(WFS))
@pytest.mark.parametrize("sd", sorted(SDS))
def test_reference_gradient_matches_finite_differences(oracle_mod, wf, sd):
    """Every weight-function family x every statistical distance; category weights, tag rules and pair weights vary
    with the case so that each kind appears with several families."""
    k = sorted(WFS).index(wf) + 4 * sorted(SDS).index(sd)
    cat_w = None if k % 2 == 0 else [0.6, 1.7, 1.1]
    tag_rule = [{"accept_same": True}, {"accept_same": False},
                {"tag_pairs": [(0, 1), (1, 2)], "accepted_pairs": True, "ordered": False}][k % 3]
    run_case(oracle_mod, [WFS[wf]], SDS[sd], cat_w, tag_rule, seed=100 + k, weighted=k % 4 == 1)


@pytest.mark.parametrize("sd", ["Hellinger", "Kullback-Leibler"])
def test_reference_gradient_per_pair_weight_functions(oracle_mod, sd):
    run_case(oracle_mod, [WFS[w] for w in sorted(WFS)], SDS[sd], [1.3, 0.4, 0.9],
             {"tag_pairs": [(0, 0), (2, 1)], "accepted_pairs": False, "ordered": True}, seed=7, per_pair_wf=True,
             weighted=True)


@pytest.mark.parametrize("sd", ["Hellinger", "Renyi"])
def test_reference_gradient_integer_kumaraswamy(oracle_mod, sd):
    """Kumaraswamy (3, 10, 2, 5) of the reference API: integer exponents (the device's powi_small path)."""
    run_case(oracle_mod, [("kumaraswamy", [3.0, 10.0, 2.0, 5.0])], SDS[sd], [0.6, 1.7, 1.1], {"accept_same": False},
             seed=81, weighted=True)


@pytest.mark.parametrize("wf", sorted(WFS))
def test_density_is_the_derivative_of_the_cdf(oracle_mod, wf):
    name, p = WFS[wf]
    xs = [0.05, 0.7, 1.6, 2.2, 3.0, 4.1, 4.99, 5.4, 7.0, 11.0]
    if name == "dagum":
        xs += [1e-6, 1e-3, 0.02]
    if name in ("uniform", "kumaraswamy"):
        xs += [p[0] + 1e-4, p[1] - 1e-4, p[0] - 1e-4, p[1] + 1e-4]   # both sides of the kinks
    for x in xs:
        h = min(1e-6, x / 4)
        num = (oracle_mod.wf_integral_point(name, p, x + h) - oracle_mod.wf_integral_point(name, p, x - h)) / (2 * h)
        got = gr.wf_density(name, p, x)
        assert abs(got - num) <= 1e-6 * max(1.0, abs(num)), (name, x, got, num)


def test_density_at_zero_and_at_the_kinks():
    assert gr.wf_density("uniform", [1.5, 5.0], 1.5) == pytest.approx(1 / 3.5)
    assert gr.wf_density("uniform", [1.5, 5.0], 5.0) == pytest.approx(1 / 3.5)
    assert gr.wf_density("uniform", [1.5, 5.0], np.nextafter(1.5, 0)) == 0.0
    assert gr.wf_density("uniform", [1.5, 5.0], np.nextafter(5.0, 9)) == 0.0
    assert gr.wf_density("kumaraswamy", [1.0, 5.5, 2.3, 1.7], np.nextafter(5.5, 9)) == 0.0
    assert gr.wf_density("dagum", [2.5, 3.0, 1.3], 0.0) == 0.0          # a p > 1
    assert gr.wf_density("dagum", [0.5, 3.0, 1.0], 0.0) == np.inf       # a p < 1
    for x in (1e-300, 1e-308, 5e-324):   # a p / x alone would overflow while the rest underflows: no inf * 0
        assert gr.wf_density("dagum", [2.5, 3.0, 1.3], x) == 0.0
    assert np.isfinite(gr.wf_density("dagum", [1.0, 3.0, 1.0], 1e-308))
