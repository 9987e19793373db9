"""MultiSurrogateOptimiser / MonoSurrogateOptimiser with the reference's surface
(optimisers.py:18-277 and :283-527) on the B200 pool-scoring path."""
from __future__ import annotations

import numpy as np

from .. import host_prep, result
from ..acquisition import spec_ehvi, spec_ehvi3d, spec_ehvi_box, spec_ei, spec_expected_decomposition
from .base import PoolOptimiserBase


class MultiSurrogateOptimiser(PoolOptimiserBase):
    """One GP per objective; default acquisition 2-D EHVI (crude 3-D EHVI for 3 objectives), or the
    expected improvement over a scalarisation when `acquisition_func` is given
    (optimisers.py:144-277).

    Additive knob `ehvi`: "reference" (default) keeps the reference's EHVI / crude 3-D EHVI above; "box" scores
    every 2 to 4 objective problem with the exact EHVI over the box decomposition (`spec_ehvi_box`)."""

    def __init__(self, test_problem, *args, ehvi="reference", **kwargs):
        if ehvi not in ("reference", "box"):
            raise ValueError(f"ehvi must be 'reference' or 'box' (got {ehvi!r})")
        super().__init__(test_problem, *args, **kwargs)
        self.ehvi = ehvi

    def _get_cached_samples(self, dimensions, sample_exponent):
        return host_prep.cached_samples(dimensions, sample_exponent, seed=int(self.rng.integers(0, 2 ** 31)))

    def solve(self, budget=100, n_init_samples=5, sample_exponent=5, acquisition_func=None):
        problem = self.test_problem
        Xsample, ysample = self._initial_design(n_init_samples)
        cached_samples = self._get_cached_samples(self.n_obj, sample_exponent)
        ref_dirs = host_prep.get_reference_directions("das-dennis", self.n_obj, n_partitions=100)
        hypervolume_convergence = []
        for _ in range(budget):
            self._update_bounds(ysample, acquisition_func)
            hypervolume_convergence.append(self._hypervolume(ysample))
            models = self._fit_models(Xsample, [ysample[:, i] for i in range(problem.n_obj)])
            ref_dir = np.asarray(ref_dirs[self.rng.integers(0, len(ref_dirs))])
            if acquisition_func is None:
                pf = self._calc_pf(ysample)
                if self.ehvi == "box":
                    spec = spec_ehvi_box(self.max_point, pf)
                elif problem.n_obj == 2:
                    spec = spec_ehvi(self.max_point, pf, cached_samples, self.semantics)
                else:
                    spec = spec_ehvi3d(self.max_point, pf, cached_samples, self.semantics)
            else:
                min_scalar = np.min([acquisition_func(y, ref_dir) for y in ysample])     # optimisers.py:250
                spec = spec_expected_decomposition(ref_dir, acquisition_func, min_scalar, cached_samples,
                                                   self.semantics)
            X_next, _ = self._propose(models, spec)
            y_next = self._objective_function(problem, X_next)
            ysample = np.vstack((ysample, y_next))
            Xsample = np.vstack((Xsample, X_next))
        mask = self._pareto_members(ysample)
        res = result.Res(ysample[mask], Xsample[mask], ysample, Xsample, hypervolume_convergence, problem.n_obj,
                         n_init_samples)
        res.timings = self.timings
        return res


class MonoSurrogateOptimiser(PoolOptimiserBase):
    """One GP on the scalarised objective, closed-form EI (optimisers.py:325-344, :373-527)."""

    def _normalize_data(self, data):
        return (data - np.min(data)) / (np.max(data) - np.min(data))

    def solve(self, aggregation_func, budget=100, n_init_samples=5):
        problem = self.test_problem
        weights = np.asarray([1 / problem.n_obj] * problem.n_obj)
        Xsample, ysample = self._initial_design(n_init_samples)
        self._update_bounds(ysample, aggregation_func)
        aggregated_samples = np.asarray([aggregation_func(y, weights) for y in ysample]).flatten()
        ref_dirs = host_prep.get_reference_directions("das-dennis", problem.n_obj, n_partitions=100)
        hypervolume_convergence = []
        for _ in range(budget):
            self._update_bounds(ysample, aggregation_func)
            hypervolume_convergence.append(self._hypervolume(ysample))
            current_best = aggregated_samples[np.argmin(aggregated_samples)]
            model = self._fit_model(Xsample, aggregated_samples)
            next_X, _ = self._propose([model], spec_ei(current_best, 0.0))
            next_y = self._objective_function(problem, next_X)
            ysample = np.vstack((ysample, next_y))
            ref_dir = ref_dirs[self.rng.integers(0, len(ref_dirs))]
            aggregated_samples = np.append(aggregated_samples, aggregation_func(next_y, ref_dir))
            Xsample = np.vstack((Xsample, next_X))
        mask = self._pareto_members(ysample)
        res = result.Res(ysample[mask], Xsample[mask], ysample, Xsample, hypervolume_convergence, problem.n_obj,
                         n_init_samples)
        res.timings = self.timings
        return res
