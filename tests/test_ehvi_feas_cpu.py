"""CPU: the constrained box EHVI (OMBO_ACQ_EHVI_BOX_FEAS) -- its spec builder, the optimiser's argument checks, the
batch closure's feasibility rule, and the Python constants against the C header."""
import os
import re

import numpy as np
import pytest

import optimobo_b200 as ob
from optimobo_b200 import _cabi
from optimobo_b200.algorithms import MultiSurrogateOptimiser

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _front():
    return np.array([[0.1, 0.9, 0.5], [0.5, 0.5, 0.5], [0.9, 0.1, 0.5]])


@pytest.mark.parametrize("c", [1, 2, 5])
def test_spec_models_and_var_eps_layout(c):
    r = np.array([1.0, 1.0, 1.0])
    spec = ob.spec_ehvi_box_feasible(r, _front(), c)
    plain = ob.spec_ehvi_box(r, _front())
    assert spec.kind == _cabi.ACQ_EHVI_BOX_FEAS == 9 and spec.n_obj == 3 and spec.n_models == 3 + c
    assert spec.var_eps == (0.0,) * 3 + (1e-5,) * c
    np.testing.assert_array_equal(spec.stripes, plain.stripes)
    np.testing.assert_array_equal(spec.cells, plain.cells)
    assert ob.spec_ehvi_box_feasible(r, _front(), c, var_eps=0.0).var_eps == (0.0,) * (3 + c)
    assert ob.spec_ehvi_box_feasible(r, _front(), c, var_eps=1e-3).var_eps[3:] == (1e-3,) * c


def test_spec_empty_front_and_front_beyond_r():
    r = [2.0, 3.0]
    for PF in (np.empty((0, 2)), [], [[2.5, 1.0], [1.0, 3.5]]):          # nothing inside r: the single box [-inf, r]
        spec = ob.spec_ehvi_box_feasible(r, PF, 2)
        np.testing.assert_array_equal(spec.stripes, [[-np.inf, 2.0], [-np.inf, 3.0]])
        np.testing.assert_array_equal(spec.cells, [[[1, 1], [0, 0]]])
        assert spec.n_models == 4
    # points beyond r drop out exactly as in the plain box spec
    PF = [[1.0, 1.0], [2.5, 0.5], [0.5, 2.0]]
    spec = ob.spec_ehvi_box_feasible(r, PF, 1)
    plain = ob.spec_ehvi_box(r, [[1.0, 1.0], [0.5, 2.0]])
    np.testing.assert_array_equal(spec.stripes, plain.stripes)
    np.testing.assert_array_equal(spec.cells, plain.cells)


def test_spec_rejects_bad_arguments():
    with pytest.raises(ValueError):
        ob.spec_ehvi_box_feasible([1, 1], _front()[:, :2], 0)
    with pytest.raises(ValueError):
        ob.spec_ehvi_box_feasible([1, 1, 1, 1], np.ones((1, 4)) * .5, 5)      # 4 + 5 > 8 models
    ob.spec_ehvi_box_feasible([1, 1, 1, 1], np.ones((1, 4)) * .5, 4)
    with pytest.raises(ValueError):
        ob.spec_ehvi_box_feasible([1, 1], _front()[:, :2], 1, var_eps=-1e-5)
    with pytest.raises(ValueError):
        ob.spec_ehvi_box_feasible([1], [[0.5]], 1)                           # the box EHVI takes 2 to 4 objectives


class _Problem:
    def __init__(self, n_obj=2, n_ieq=2, n_eq=0):
        self.n_var, self.n_obj, self.n_ieq_constr, self.n_eq_constr = 2, n_obj, n_ieq, n_eq
        self.xl, self.xu = np.zeros(2), np.ones(2)


def test_optimiser_argument_checks():
    MultiSurrogateOptimiser(_Problem(), ehvi="box", constrained=True)
    MultiSurrogateOptimiser(_Problem(n_obj=4, n_ieq=4), ehvi="box", constrained=True)
    MultiSurrogateOptimiser(_Problem(), constrained=False)                   # the default loop needs nothing
    with pytest.raises(ValueError, match="ehvi='box'"):
        MultiSurrogateOptimiser(_Problem(), constrained=True)
    with pytest.raises(ValueError, match="inequality constraints only"):
        MultiSurrogateOptimiser(_Problem(n_eq=1), ehvi="box", constrained=True)
    with pytest.raises(ValueError, match="at least one"):
        MultiSurrogateOptimiser(_Problem(n_ieq=0), ehvi="box", constrained=True)
    with pytest.raises(ValueError, match="<= 8"):
        MultiSurrogateOptimiser(_Problem(n_obj=3, n_ieq=6), ehvi="box", constrained=True)
    opt = MultiSurrogateOptimiser(_Problem(), ehvi="box", constrained=True)
    with pytest.raises(ValueError, match="acquisition_func"):
        opt.solve(budget=1, acquisition_func=lambda y, w: 0.0)
    assert not MultiSurrogateOptimiser(_Problem(), ehvi="box").constrained


def test_batch_spec_for_feasibility_rule():
    opt = MultiSurrogateOptimiser(_Problem(), [0, 0], [1.0, 1.0], ehvi="box", constrained=True, prep_on_device=False)
    pf = np.array([[0.2, 0.8], [0.8, 0.2]])
    spec_for = opt._constrained_spec_for(pf)

    def same(spec, front):
        want = ob.spec_ehvi_box_feasible([1.0, 1.0], front, 2)
        assert spec.kind == _cabi.ACQ_EHVI_BOX_FEAS and spec.n_models == 4 and spec.var_eps == want.var_eps
        np.testing.assert_array_equal(spec.stripes, want.stripes)
        np.testing.assert_array_equal(spec.cells, want.cells)

    same(spec_for(np.empty((0, 4))), pf)
    rows = np.array([
        [0.5, 0.5, -0.1, -2.0],     # feasible, inside r, non-dominated: joins the front
        [0.1, 0.1, 0.3, -1.0],      # one constraint > 0: stays out although it would dominate everything
        [0.1, 0.1, -1.0, 1e-9],     # the other constraint just above 0: stays out
        [1.5, 0.05, -1.0, -1.0],    # feasible but beyond r: stays out
        [0.6, 0.6, 0.0, 0.0],       # feasible at the boundary (<= 0), dominated by the first row: no change
    ])
    same(spec_for(rows), np.array([[0.2, 0.8], [0.8, 0.2], [0.5, 0.5]]))
    same(spec_for(rows[1:4]), pf)
    # an empty feasible front takes the first feasible believed row
    spec_for = opt._constrained_spec_for(np.empty((0, 2)))
    same(spec_for(rows[1:4]), np.empty((0, 2)))
    same(spec_for(rows[4:]), rows[4:, :2])


def test_cabi_matches_header():
    header = open(os.path.join(ROOT, "include", "optimobo_b200.h")).read()
    kinds = dict((k, int(v)) for k, v in re.findall(r"OMBO_ACQ_(\w+)\s*=\s*(\d+)", header))
    assert kinds["EHVI_BOX_FEAS"] == _cabi.ACQ_EHVI_BOX_FEAS == 9
    assert kinds["EHVI_BOX"] == _cabi.ACQ_EHVI_BOX == 8
    assert int(re.search(r"#define OMBO_MAX_GP\s+(\d+)", header).group(1)) == _cabi.MAX_GP
    assert int(re.search(r"#define OMBO_ABI_VERSION\s+(\d+)", header).group(1)) == 1


def test_feasible_kind_is_never_certified():
    from optimobo_b200.acquisition import _certifiable
    assert _certifiable(ob.spec_ehvi_box([1, 1], [[0.5, 0.5]]))
    assert not _certifiable(ob.spec_ehvi_box_feasible([1, 1], [[0.5, 0.5]], 1))
