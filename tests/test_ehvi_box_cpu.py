"""CPU: the box decomposition behind the exact k-objective EHVI (host_prep.ehvi_boxes) against the hypervolume, the
grid oracle against the box sum, and closed-form anchors.  No GPU needed."""
import numpy as np
import pytest

from optimobo_b200 import host_prep as H
from oracle import oracle as O
from ehvi_oracle import ehvi_grid_batched, expected_shortfall


def _corners(table, boxes):
    k = table.shape[0]
    U = np.stack([table[i, boxes[:, 0, i]] for i in range(k)], axis=1)
    L = np.stack([table[i, boxes[:, 1, i]] for i in range(k)], axis=1)
    return L, U


def _box_ehvi(table, boxes, mu, sd):
    """numpy sum over the boxes: EHVI[m] = sum_c prod_i (H_i(u_ci) - H_i(l_ci))."""
    L, U = _corners(table, boxes)
    out = np.ones((len(mu), len(boxes)))
    for i in range(table.shape[0]):
        out *= (expected_shortfall(U[None, :, i], mu[:, i:i + 1], sd[:, i:i + 1])
                - expected_shortfall(L[None, :, i], mu[:, i:i + 1], sd[:, i:i + 1]))
    return out.sum(1)


def _sphere(P, k, rng):
    X = np.abs(rng.normal(size=(P, k)))
    return X / np.linalg.norm(X, axis=1, keepdims=True)


def _fronts(k):
    """(PF, r) cases: random fronts with duplicates, points beyond r, coordinates equal to r, and the empty front."""
    rng = np.random.default_rng(100 + k)
    out = []
    for P in (1, 2, 7, 25, 60):
        F = _sphere(P, k, rng)
        r = np.full(k, 1.05)
        out.append((F, r))
    F = _sphere(30, k, rng)
    F = np.vstack([F, F[:5]])                                  # duplicates
    F = np.vstack([F, F[5:8] + 2.0])                           # beyond r
    r = F[:30].max(0) + 0.01
    F[10, 0] = r[0]                                            # coordinate equal to r
    out.append((F, r))
    Q = rng.integers(0, 4, size=(40, k)).astype(float)        # heavy ties on a lattice
    out.append((Q, np.full(k, 4.0)))
    out.append((np.empty((0, k)), np.ones(k)))                 # empty front
    return out


@pytest.mark.parametrize("k", [2, 3, 4])
def test_decomposition_tiles_the_free_region(k):
    for PF, r in _fronts(k):
        table, boxes = H.ehvi_boxes(PF, r)
        B = table.shape[1]
        assert table.shape == (k, B) and boxes.shape[1:] == (2, k) and boxes.dtype.kind == "i"
        assert np.all(np.isneginf(table[:, 0])) and np.all(table[:, -1] == r)
        assert np.all(np.diff(table[:, 1:], axis=1) >= 0)
        assert np.all(boxes[:, 0] > boxes[:, 1]) and boxes.min() >= 0 and boxes.max() < B
        L, U = _corners(table, boxes)
        lo = np.minimum(np.asarray(PF).reshape(-1, k).min(0) if len(PF) else r, r) - 0.5
        vol = np.prod(np.clip(U - np.maximum(L, lo), 0, None), axis=1).sum()
        full = np.prod(r - lo)
        np.testing.assert_allclose(vol + H.hypervolume(PF, r), full, rtol=1e-12)
        if len(PF) == 0:
            assert boxes.shape[0] == 1 and np.array_equal(boxes[0, 1], np.zeros(k))


@pytest.mark.parametrize("k", [2, 3, 4])
def test_box_hvi_equals_hypervolume_difference(k):
    rng = np.random.default_rng(7 + k)
    for PF, r in _fronts(k):
        table, boxes = H.ehvi_boxes(PF, r)
        L, U = _corners(table, boxes)
        base = H.hypervolume(PF, r)
        P = np.asarray(PF).reshape(-1, k)
        lo = (P.min(0) if len(P) else r) - 0.3
        Y = rng.uniform(lo, r + 0.1, size=(200, k))
        Y[:20] = P[rng.integers(0, len(P), 20)] if len(P) else Y[:20]      # some y on the front itself
        for y in Y:
            hvi = np.prod(np.clip(U - np.maximum(L, y), 0, None), axis=1).sum()
            want = H.hypervolume(np.vstack([P, y]), r) - base
            assert abs(hvi - want) <= 1e-12 * max(1.0, np.prod(r - lo)), (hvi, want)


@pytest.mark.parametrize("k", [2, 3, 4])
def test_grid_oracle_equals_box_sum(k):
    rng = np.random.default_rng(20 + k)
    for PF, r in _fronts(k):
        table, boxes = H.ehvi_boxes(PF, r)
        P = np.asarray(PF).reshape(-1, k)
        center = P[rng.integers(0, len(P), 64)] if len(P) else np.tile(r - 0.5, (64, 1))
        mu = center + rng.normal(0, 0.1, size=(64, k))
        sd = rng.uniform(0.01, 0.3, size=(64, k))
        got = ehvi_grid_batched(mu, sd ** 2, PF, r)
        want = _box_ehvi(table, boxes, mu, sd)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12 * np.abs(want).max())


def test_anchor_2d():
    PF = np.array([[.1, .9], [.4, .5], [.8, .2]])
    mu, sd = np.array([[.3, .6]]), np.array([[.2, .3]])
    table, boxes = H.ehvi_boxes(PF, [1, 1])
    np.testing.assert_allclose(_box_ehvi(table, boxes, mu, sd), [0.0768782210398855], rtol=1e-14)
    np.testing.assert_allclose(ehvi_grid_batched(mu, sd ** 2, PF, [1, 1]), [0.0768782210398855], rtol=1e-14)


def test_anchor_2d_golden(golden):
    mu, var = golden["acq_in_mu2"], golden["acq_in_var2"]
    PF, r = golden["acq_out_calc_pf"], golden["acq_in_ref"]
    want = O.ehvi2d_aux_batched(PF, r, mu[:, 0], mu[:, 1], np.sqrt(var[:, 0]), np.sqrt(var[:, 1]), exact=True)
    table, boxes = H.ehvi_boxes(PF, r)
    np.testing.assert_allclose(_box_ehvi(table, boxes, mu, np.sqrt(var)), want, rtol=1e-10,
                               atol=1e-13 * np.abs(want).max())
    np.testing.assert_allclose(ehvi_grid_batched(mu, var, PF, r), want, rtol=1e-10, atol=1e-13 * np.abs(want).max())


def test_anchor_single_point_3d():
    """One front point p: EHVI = prod H_i(r_i) - prod (H_i(r_i) - H_i(p_i))."""
    p, r = np.array([0.3, 0.5, 0.2]), np.array([1.0, 1.2, 0.9])
    rng = np.random.default_rng(5)
    mu = rng.uniform(0, 1, size=(50, 3))
    sd = rng.uniform(0.05, 0.5, size=(50, 3))
    Hr = expected_shortfall(r[None, :], mu, sd)
    Hp = expected_shortfall(p[None, :], mu, sd)
    want = Hr.prod(1) - (Hr - Hp).prod(1)
    table, boxes = H.ehvi_boxes(p[None, :], r)
    np.testing.assert_allclose(_box_ehvi(table, boxes, mu, sd), want, rtol=1e-12)
    np.testing.assert_allclose(ehvi_grid_batched(mu, sd ** 2, p[None, :], r), want, rtol=1e-12)


def test_anchor_sigma_to_zero_is_hvi():
    rng = np.random.default_rng(9)
    PF = _sphere(30, 3, rng)
    r = np.full(3, 1.1)
    table, boxes = H.ehvi_boxes(PF, r)
    mu = rng.uniform(0.2, 1.1, size=(40, 3))
    base = H.hypervolume(PF, r)
    want = np.array([H.hypervolume(np.vstack([PF, y]), r) - base for y in mu])
    got = ehvi_grid_batched(mu, np.full_like(mu, 1e-24), PF, r)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(_box_ehvi(table, boxes, mu, np.full_like(mu, 1e-12)), want, rtol=1e-9, atol=1e-12)


def c4_front():
    """The C4 shape: DTLZ2, n = 512, d = 12, seed 4, r = Y.max(0) + 0.1."""
    rng = np.random.default_rng(4)
    X = rng.random((512, 12))
    g = ((X[:, 2:] - .5) ** 2).sum(1)
    a, b = .5 * np.pi * X[:, 0], .5 * np.pi * X[:, 1]
    Y = np.column_stack([(1 + g) * np.cos(a) * np.cos(b), (1 + g) * np.cos(a) * np.sin(b), (1 + g) * np.sin(a)])
    return H.calc_pf(Y), Y.max(0) + 0.1


def test_monte_carlo_c4():
    PF, r = c4_front()
    table, boxes = H.ehvi_boxes(PF, r)
    L, U = _corners(table, boxes)
    mu, sd = PF.mean(0) - 0.05, np.array([.1, .15, .2])
    e = _box_ehvi(table, boxes, mu[None, :], sd[None, :])[0]
    rng = np.random.default_rng(11)
    S = rng.normal(mu, sd, size=(20000, 3))
    hvi = np.array([np.prod(np.clip(U - np.maximum(L, s), 0, None), axis=1).sum() for s in S])
    se = hvi.std() / np.sqrt(len(hvi))
    assert abs(e - hvi.mean()) < 4 * se, (e, hvi.mean(), se)
    np.testing.assert_allclose(ehvi_grid_batched(mu[None, :], sd[None, :] ** 2, PF, r), [e], rtol=1e-12)


def test_input_checks():
    with pytest.raises(ValueError):
        H.ehvi_boxes(np.zeros((3, 5)), np.ones(5))
    with pytest.raises(ValueError):
        H.ehvi_boxes(np.zeros((3, 1)), np.ones(1))
