"""CPU: the hypervolume-based probability of improvement over the box decomposition (tests/hv_poi_oracle.py) against
the reference's 2-D cells, against the grid brute force for 3 and 4 objectives, and the spec it is scored from
(acquisition.spec_hv_poi_box on the host).  No GPU needed."""
import numpy as np
import pytest

import optimobo_b200 as ob
from optimobo_b200 import _cabi, host_prep as H
from oracle import oracle as O
from hv_poi_oracle import hv_poi_box_batched, hv_poi_grid_batched, region_ref


def _random_2d(rng):
    """A random 2-D front with the ideal at or below it and max_point on either side of its maximum."""
    Y = rng.random((int(rng.integers(1, 30)), 2))
    PF = H.calc_pf(Y)
    ideal = Y.min(0) - rng.random(2) * 0.1
    maxp = Y.max(0) + rng.random(2) * 0.3 - 0.15
    return PF, ideal, maxp


def test_box_oracle_equals_reference_cells_2d():
    rng = np.random.default_rng(0)
    below = above = 0
    for _ in range(200):
        PF, ideal, maxp = _random_2d(rng)
        below += np.any(maxp < PF.max(0))
        above += np.any(maxp > PF.max(0))
        cells = H.decompose_into_cells(PF, ideal, maxp)
        mu = rng.random((64, 2)) * 1.4 - 0.2
        var = rng.random((64, 2)) * 0.05
        want = O.hv_poi_batched(mu, var, cells)
        # the reference subtracts two Phi near 1 for a cell above the mean and loses ~1e-16 absolute there, which the
        # box oracle does not: values below ~1e-4 differ by up to that much
        np.testing.assert_allclose(hv_poi_box_batched(mu, var, PF, ideal, maxp), want, rtol=1e-12, atol=1e-16)
    assert below > 20 and above > 100


def test_box_oracle_equals_reference_cells_golden(golden):
    PF, ideal, maxp = golden["acq_out_calc_pf"], golden["emo_in_ideal"], golden["emo_in_max"]
    mu, var = golden["acq_in_mu2"], golden["acq_in_var2"]
    assert np.all(PF >= ideal)
    want = O.hv_poi_batched(mu, var, H.decompose_into_cells(PF, ideal, maxp))
    np.testing.assert_allclose(hv_poi_box_batched(mu, var, PF, ideal, maxp), want, rtol=1e-12, atol=1e-16)
    np.testing.assert_allclose(want, golden["emo_out_poi"], rtol=1e-12, atol=0)


@pytest.mark.parametrize("k", [2, 3, 4])
def test_box_oracle_equals_grid_oracle(k):
    rng = np.random.default_rng(30 + k)
    for trial in range(8):
        Y = rng.random((12, k))
        PF = H.calc_pf(Y)
        ideal = Y.min(0) - (0.05 if trial % 2 else 0.0)
        maxp = Y.max(0) + rng.random(k) * 0.3 - 0.1
        if trial == 7:
            PF = np.vstack([PF, PF[:2], PF[0] + 0.01])            # duplicates and a dominated point
        mu = rng.random((40, k)) * 1.2 - 0.1
        var = rng.random((40, k)) * 0.05
        mu[:4] = ideal - 0.5                                      # far below every box
        mu[4:8] = region_ref(PF, maxp) + 0.1                      # beyond r': no volume above the mean
        want = hv_poi_grid_batched(mu, var, PF, ideal, maxp)
        got = hv_poi_box_batched(mu, var, PF, ideal, maxp)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
        assert np.all(want[4:8] == 0) and np.all(want[:4] > 0) and want.max() > 0


def test_empty_front_is_one_box():
    ideal, maxp = np.array([0.1, 0.2, 0.0]), np.array([1.0, 1.5, 0.7])
    mu, var = np.array([[0.5, 0.5, 0.3], [2.0, 0.5, 0.3]]), np.full((2, 3), 0.02)
    from scipy.special import ndtr
    sd = np.sqrt(var + 1e-5)
    poi = np.prod(ndtr((maxp - mu) / sd) - ndtr((ideal - mu) / sd), 1)
    imp = np.prod(np.clip(maxp - np.maximum(ideal, mu), 0, None), 1)
    np.testing.assert_allclose(hv_poi_box_batched(mu, var, np.empty((0, 3)), ideal, maxp), poi * imp, rtol=1e-14)
    np.testing.assert_allclose(hv_poi_grid_batched(mu, var, np.empty((0, 3)), ideal, maxp), poi * imp, rtol=1e-14)
    spec = ob.spec_hv_poi_box(ideal, maxp, np.empty((0, 3)))
    np.testing.assert_array_equal(spec.stripes, np.column_stack([ideal, maxp]))
    np.testing.assert_array_equal(spec.cells, [[[1, 1, 1], [0, 0, 0]]])


@pytest.mark.parametrize("k", [3, 4])
def test_permuting_objectives(k):
    rng = np.random.default_rng(40 + k)
    Y = rng.random((15, k))
    PF, ideal, maxp = H.calc_pf(Y), Y.min(0), Y.max(0) + 0.05
    mu, var = rng.random((30, k)), rng.random((30, k)) * 0.05
    base = hv_poi_box_batched(mu, var, PF, ideal, maxp)
    for _ in range(4):
        p = rng.permutation(k)
        np.testing.assert_allclose(hv_poi_box_batched(mu[:, p], var[:, p], PF[:, p], ideal[p], maxp[p]), base,
                                   rtol=1e-12, atol=0)


def test_spec_table_is_clamped_at_the_ideal():
    rng = np.random.default_rng(5)
    Y = rng.random((20, 3))
    PF = H.calc_pf(Y)
    ideal = Y.min(0) + np.array([0.0, 0.1, -0.2])                 # above some front coordinates in objective 1
    maxp = Y.max(0) - np.array([0.1, 0.0, -0.1])                  # below the front's maximum in objective 0
    spec = ob.spec_hv_poi_box(ideal, maxp, PF)
    r = np.maximum(maxp, PF.max(0))
    table, boxes = H.ehvi_boxes(PF, r)
    assert spec.kind == _cabi.ACQ_HV_POI_BOX and spec.n_obj == 3 and spec.n_models == 3
    assert spec.var_eps == (1e-5,) * 3 and spec.ref == tuple(r)
    np.testing.assert_array_equal(spec.stripes, np.maximum(table, ideal[:, None]))
    np.testing.assert_array_equal(spec.cells, boxes)
    assert np.all(spec.stripes[:, 0] == ideal) and np.all(spec.stripes[:, -1] == r)
    assert np.all(np.diff(spec.stripes, axis=1) >= 0)
    a = spec.c_struct("cpu")
    assert a.n_pf == table.shape[1] and a.n_cells == len(boxes)


def test_spec_input_checks():
    PF = np.array([[0.2, 0.8, 0.5], [0.8, 0.2, 0.5]])
    ob.spec_hv_poi_box([0, 0, 0], [1, 1, 1], PF)
    for ideal, maxp, F in (([0] * 5, [1] * 5, np.zeros((2, 5))),        # k = 5
                           ([0], [1], np.zeros((2, 1))),                # k = 1
                           ([0, 0], [1, 1, 1], PF),                     # ideal of the wrong length
                           ([0, np.nan, 0], [1, 1, 1], PF),
                           ([0, 0, 0], [1, np.inf, 1], PF),
                           ([0, 0, 0], [1, 1, 1], np.vstack([PF, [0.1, -np.inf, 0.3]]))):
        with pytest.raises(ValueError):
            ob.spec_hv_poi_box(ideal, maxp, F)


def test_emo_rejects_more_than_four_objectives():
    from optimobo_b200.algorithms import EMO

    class _P:
        def __init__(self, k):
            self.n_var, self.n_obj, self.xl, self.xu = 2, k, np.zeros(2), np.ones(2)

    for k in (3, 4):
        EMO(_P(k), None, None)
    for k in (1, 5):
        with pytest.raises(ValueError):
            EMO(_P(k), None, None)
