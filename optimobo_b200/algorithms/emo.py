"""EMO (emo.py:14-333): hypervolume-based probability of improvement over the non-dominated region.  Two
objectives score over the reference's cell decomposition (emo.py:21 stops there); three and four score the same
quantity over the box decomposition (`spec_hv_poi_box`), which the reference does not have."""
from __future__ import annotations

import numpy as np

from .. import host_prep, result
from ..acquisition import spec_hv_poi, spec_hv_poi_box
from .base import PoolOptimiserBase


class EMO(PoolOptimiserBase):
    def __init__(self, test_problem, ideal_point, max_point, **kw):
        super().__init__(test_problem, ideal_point, max_point, **kw)
        if not 2 <= self.n_obj <= 4:
            raise ValueError(f"EMO scores 2 to 4 objectives (got {self.n_obj})")

    def decompose_into_cells(self, data_points):
        if self._prep_device(len(data_points)):
            from .. import device_prep
            return device_prep.decompose_into_cells(data_points, self.ideal_point, self.max_point,
                                                    self.device).cpu().numpy()
        return host_prep.decompose_into_cells(data_points, self.ideal_point, self.max_point)

    def _spec(self, pf):
        if self.n_obj == 2:
            return spec_hv_poi(self.decompose_into_cells(pf))
        return spec_hv_poi_box(self.ideal_point, self.max_point, pf, device=self._box_device(pf))

    def solve(self, budget=100, n_init_samples=5):
        problem = self.test_problem
        Xsample, ysample = self._initial_design(n_init_samples)
        hypervolume_convergence = []
        for _ in range(budget):
            self._update_bounds(ysample)
            hypervolume_convergence.append(self._hypervolume(ysample))
            models = self._fit_models(Xsample, [ysample[:, i] for i in range(self.n_obj)])
            X_next, _ = self._propose(models, self._spec(self._calc_pf(ysample)))
            y_next = self._objective_function(problem, X_next)
            ysample = np.vstack((ysample, y_next))
            Xsample = np.vstack((Xsample, X_next))
        mask = self._pareto_members(ysample)
        res = result.Res(ysample[mask], Xsample[mask], ysample, Xsample, hypervolume_convergence, problem.n_obj,
                         n_init_samples)
        res.timings = self.timings
        return res
