"""CPU: the device box decomposition's Python surface -- the wrapper's argument checks (raised before any device
work), the optimiser's host / device selection rule, the spec builders' default host path and the new header
constants."""
import os
import re

import numpy as np
import pytest

import optimobo_b200 as ob
from optimobo_b200 import _cabi, device_prep
from optimobo_b200.algorithms import MultiSurrogateOptimiser
from optimobo_b200.algorithms import optimisers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("PF,r,match", [
    (np.ones((2, 1)) * .5, [1.0], "2 to 4 objectives"),
    (np.ones((2, 5)) * .5, [1.0] * 5, "2 to 4 objectives"),
    (np.ones((2, 3)) * .5, [1.0, np.inf, 1.0], "finite"),
    (np.ones((2, 3)) * .5, [1.0, np.nan, 1.0], "finite"),
    (np.ones((2, 2)) * .5, [1.0] * 3, r"\(p, 3\)"),
    (np.ones((2, 3, 1)) * .5, [1.0] * 3, r"\(p, 3\)"),
    (np.ones(7) * .5, [1.0] * 3, r"\(p, 3\)"),
    (np.ones((16385, 2)) * .5, [1.0] * 2, "16384"),
])
def test_wrapper_argument_checks(PF, r, match):
    with pytest.raises(ValueError, match=match):
        device_prep.ehvi_boxes(PF, r, "cuda:0")


class _Problem:
    def __init__(self, n_obj=3):
        self.n_var, self.n_obj, self.n_ieq_constr, self.n_eq_constr = 2, n_obj, 0, 0
        self.xl, self.xu = np.zeros(2), np.ones(2)


@pytest.mark.parametrize("prep", [True, False, "auto"])
def test_selection_rule(prep):
    opt = MultiSurrogateOptimiser(_Problem(), ehvi="box", prep_on_device=prep, device="cuda:1")
    lo, hi = optimisers.BOX_DEVICE_MIN_FRONT, optimisers.BOX_DEVICE_MAX_FRONT
    assert hi == _cabi.EHVI_BOX_MAX_BREAKS - 2
    rng = np.random.default_rng(0)
    for n in (0, 1, lo - 1, lo, hi, hi + 1):
        front = rng.random((n, 3))
        want = prep is True or (prep == "auto" and n >= lo)
        assert opt._box_device(front) == ("cuda:1" if want and n <= hi else None), (prep, n)
        if n:
            for bad in (np.nan, np.inf, -np.inf):                             # a non-finite front stays on the host
                f = front.copy()
                f[n // 2, 1] = bad
                assert opt._box_device(f) is None


def test_spec_default_stays_on_the_host():
    PF, r = np.array([[0.2, 0.8, 0.5], [0.8, 0.2, 0.5]]), [1.0, 1.0, 1.0]
    for spec in (ob.spec_ehvi_box(r, PF), ob.spec_ehvi_box(r, PF, device=None),
                 ob.spec_ehvi_box_feasible(r, PF, 2), ob.spec_ehvi_box_feasible(r, PF, 2, device=None)):
        table, boxes = ob.host_prep.ehvi_boxes(PF, r)
        assert isinstance(spec.stripes, np.ndarray) and isinstance(spec.cells, np.ndarray)
        assert spec.cells.dtype == np.float64
        np.testing.assert_array_equal(spec.stripes, table)
        np.testing.assert_array_equal(spec.cells, boxes)


def test_cabi_matches_header():
    header = open(os.path.join(ROOT, "include", "optimobo_b200.h")).read()
    assert int(re.search(r"#define OMBO_ERR_SPACE\s+(-\d+)", header).group(1)) == _cabi.ERR_SPACE == -5
    assert int(re.search(r"#define OMBO_ERR_UNSUPPORTED\s+(-\d+)", header).group(1)) == _cabi.ERR_UNSUPPORTED
    assert int(re.search(r"#define OMBO_EHVI_BOX_MAX_BREAKS\s+(\d+)", header).group(1)) == _cabi.EHVI_BOX_MAX_BREAKS
    assert re.search(r"int ombo_ehvi_boxes\(", header) and "ombo_ehvi_boxes" in _cabi.EXPORTS
    assert int(re.search(r"#define OMBO_ABI_VERSION\s+(\d+)", header).group(1)) == 1
