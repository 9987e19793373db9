"""CPU: the 50-digit reference (tests/acq_mpmath.py) against the float64 restatement (oracle/oracle.py) where the
float64 formulas are well conditioned, against the SURVEY section 8c anchors, and the properties the kernels are held
to (non-negative values, EI monotone in `best`, EI above the improvement of the mean)."""
import numpy as np
import pytest

import acq_mpmath as M
from ehvi_oracle import ehvi_grid_batched
from oracle import oracle as O

TIGHT = 1e-12


def close(a, b, rtol=TIGHT, atol=0.0):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def _front(P, rng):
    t = np.sort(rng.random(P))
    return np.column_stack([t, 1.0 - np.sqrt(t)])


# ------------------------------------------------------------------------------------------
# agreement with the float64 oracle where it is well conditioned
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("var_eps", [0.0, 1e-6])
def test_ei_matches_oracle_for_moderate_g(var_eps):
    rng = np.random.default_rng(1)
    var = rng.uniform(0.01, 4.0, 400)
    g = rng.uniform(-5.0, 5.0, 400)
    best = 0.3
    mu = best - g * np.sqrt(var + var_eps)
    close(M.expected_improvement(mu, var, best, var_eps), O.expected_improvement(mu, var, best, var_eps))
    close(M.pareto_ei(mu[::-1], mu, var, best), O.pareto_ei(mu[::-1], mu, var, best))


def test_pof_and_constrained_ei_match_oracle():
    rng = np.random.default_rng(2)
    mu = np.column_stack([rng.uniform(-1, 1, 300), rng.uniform(-2, 2, (300, 2))])
    var = rng.uniform(0.05, 2.0, (300, 3))
    close(M.probability_of_feasibility(mu[:, 1], var[:, 1]), O.probability_of_feasibility(mu[:, 1], var[:, 1]))
    close(M.constrained_ei(mu, var, 0.2), O.constrained_ei(mu, var, 0.2))


def test_hv_poi_matches_oracle_near_the_cells():
    rng = np.random.default_rng(3)
    cells = O.decompose_into_cells_2d(_front(6, rng), [0.0, 0.0], [1.0, 1.0])
    mu = rng.uniform(0.0, 1.0, (200, 2))
    var = rng.uniform(0.01, 0.2, (200, 2))
    close(M.hv_poi(mu, var, cells), O.hv_poi_batched(mu, var, cells), rtol=1e-11)


@pytest.mark.parametrize("semantics", ["reference", "exact"])
def test_ehvi2d_matches_oracle(semantics):
    rng = np.random.default_rng(4)
    PF, r = _front(7, rng), np.array([1.1, 1.1])
    y1, y2 = O.ehvi_stripes(PF, r)
    mu = rng.uniform(0.0, 1.0, (150, 2))
    var = rng.uniform(0.02, 0.3, (150, 2))
    cache_c = (1.02, 0.03)
    got = M.ehvi2d_posterior(np.stack([y1, y2]), mu, var, semantics, cache_c)
    if semantics == "reference":
        want = O.ehvi2d_aux_batched(PF, r, mu[:, 0], mu[:, 1], var[:, 0] * cache_c[0], var[:, 0] * cache_c[1])
    else:
        want = O.ehvi_batched(mu[:, 0], mu[:, 1], var[:, 0], var[:, 1], PF, r, None, "exact")
    close(got, want, rtol=1e-11, atol=1e-14 * np.abs(want).max())


def test_ehvi3d_matches_oracle():
    rng = np.random.default_rng(5)
    cache = rng.normal(size=(32, 3))
    PF = np.abs(rng.normal(size=(12, 3)))
    PF /= np.linalg.norm(PF, axis=1, keepdims=True)
    r = PF.max(0) + 0.2
    sminus = O.hypervolume(PF, r)
    mu = PF[rng.integers(0, 12, 60)] - rng.uniform(0.0, 0.3, (60, 3))
    var = rng.uniform(0.005, 0.05, (60, 3))
    for sem in ("reference", "exact"):
        want = O.ehvi3d_batched(mu, var, r, sminus, cache, sem)
        assert (want > 0).sum() > 20
        close(M.ehvi3d(mu, var, r, sminus, cache, sem), want, rtol=1e-12, atol=1e-15)


def test_ehvi_box_matches_grid_oracle():
    from optimobo_b200 import host_prep     # pure numpy: the boxes under test come from the package's decomposition
    rng = np.random.default_rng(6)
    for k in (2, 3):
        PF = np.abs(rng.normal(size=(8, k)))
        PF /= np.linalg.norm(PF, axis=1, keepdims=True)
        r = PF.max(0) + 0.1
        table, boxes = host_prep.ehvi_boxes(PF, r)
        mu = PF[rng.integers(0, 8, 40)] + rng.normal(0, 0.05, (40, k))
        var = rng.uniform(0.001, 0.01, (40, k))
        want = ehvi_grid_batched(mu, var, PF, r)
        close(M.ehvi_box(table, boxes, mu, var), want, rtol=1e-10, atol=1e-14 * np.abs(want).max())


# ------------------------------------------------------------------------------------------
# SURVEY section 8c anchors (the same constants test_oracle_golden.py::test_anchors pins)
# ------------------------------------------------------------------------------------------
def test_anchors():
    PF = np.array([[.1, .9], [.4, .5], [.8, .2]])
    st = np.stack(O.ehvi_stripes(PF, [1.0, 1.0]))
    close(M.ehvi2d(st, [.3], [.6], [.2], [.3], exact=False), [0.0700010532552525])
    close(M.ehvi2d(st, [.3], [.6], [.2], [.3], exact=True), [0.0768782210398855])
    close(M.expected_improvement([.5], [.04], .6), [0.13955931], rtol=1e-7)
    close(M.expected_improvement([.5], [.04], .6, 1e-6), [0.13956019], rtol=1e-7)
    close(M.constrained_ei(np.array([[.5, -.1, .2]]), np.array([[.04, .01, .02]]), .6), [0.0092396], rtol=1e-5)
    close(M.pareto_ei([.7], [.5], [.04], .6), [0.09769213], rtol=1e-7)
    cells = O.decompose_into_cells_2d(PF, [0, 0], [1, 1])
    close(M.hv_poi(np.array([[.3, .6]]), np.array([[.04, .09]]), cells), [0.018681436421498922], rtol=1e-9)


# ------------------------------------------------------------------------------------------
# the properties the kernels are held to
# ------------------------------------------------------------------------------------------
def test_values_are_never_negative_in_the_tails():
    g = np.linspace(-40.0, 40.0, 321)
    ei = M.expected_improvement(-g, np.ones_like(g), 0.0)
    assert np.all(ei >= 0)
    assert np.all(ei[g >= -37.0] > 0)                  # a normal double down to g ~ -37
    pof = M.probability_of_feasibility(np.linspace(-15, 15, 101), np.full(101, 0.25))
    assert np.all(pof >= 0) and pof[-1] > 0 and pof[0] == 1.0
    cei = M.constrained_ei(np.array([[0.0, 3.2, 3.2], [0.0, 5.0, 5.0]]), np.array([[1.0, 0.1, 0.1]] * 2), 0.0)
    assert np.all(cei > 0)
    close(cei[0], M.expected_improvement([0.0], [1.0], 0.0)[0] * M.probability_of_feasibility([3.2], [0.1])[0] ** 2,
          rtol=1e-14)
    cells = np.array([[[1.0, 1.0], [0.0, 0.0]], [[2.0, 0.5], [1.0, 0.0]]])
    poi = M.hv_poi(np.array([[-0.3, -0.3], [3.0, 3.0], [0.5, 0.5]]), np.full((3, 2), 0.01), cells)
    assert np.all(poi >= 0) and poi[0] > 0
    PF = np.array([[.1, .9], [.4, .5], [.8, .2]])
    st = np.stack(O.ehvi_stripes(PF, [1.0, 1.0]))
    mu = np.array([[1.0, 1.0], [0.9, 0.95], [0.5, 0.6], [5.0, 5.0]])
    ex = M.ehvi2d_posterior(st, mu, np.full((4, 2), 1e-3), "exact")
    assert np.all(ex >= 0) and ex[1] > 0


def test_ei_non_decreasing_in_best():
    rng = np.random.default_rng(7)
    mu, var = rng.normal(size=60), rng.uniform(1e-4, 1.0, 60)
    prev = M.expected_improvement(mu, var, -30.0)
    for best in np.linspace(-30.0, 30.0, 25)[1:]:
        cur = M.expected_improvement(mu, var, best)
        assert np.all(cur >= prev)
        prev = cur


def test_ei_above_the_improvement_of_the_mean():
    """EI >= (best - mu)^+ s / (s + 1e-10): Jensen's bound scaled by the formula's 1e-10 guard in the denominator.
    The plain bound (best - mu)^+ fails at the variance floor, where s ~ 3e-8 is not large against 1e-10."""
    rng = np.random.default_rng(8)
    mu = rng.normal(size=80)
    for var in (np.full(80, 1e-15), rng.uniform(1e-15, 1e-9, 80), rng.uniform(0.01, 1.0, 80)):
        s = np.sqrt(var)
        ei = M.expected_improvement(mu, var, 0.1)
        bound = np.maximum(0.1 - mu, 0.0) * (s / (s + 1e-10))
        assert np.all(ei >= bound * (1 - 1e-15))
    var = np.full(80, 1e-15)
    assert np.any(M.expected_improvement(mu, var, 0.1) < np.maximum(0.1 - mu, 0.0))

