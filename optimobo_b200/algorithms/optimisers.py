"""MultiSurrogateOptimiser / MonoSurrogateOptimiser with the reference's surface
(optimisers.py:18-277 and :283-527) on the B200 pool-scoring path."""
from __future__ import annotations

import numpy as np

from .. import host_prep, result
from ..acquisition import (spec_ehvi, spec_ehvi3d, spec_ehvi_box, spec_ehvi_box_feasible, spec_ei,
                           spec_expected_decomposition)
from .base import BOX_DEVICE_MAX_FRONT, BOX_DEVICE_MIN_FRONT, PoolOptimiserBase  # noqa: F401


class MultiSurrogateOptimiser(PoolOptimiserBase):
    """One GP per objective; default acquisition 2-D EHVI (crude 3-D EHVI for 3 objectives), or the
    expected improvement over a scalarisation when `acquisition_func` is given
    (optimisers.py:144-277).

    Additive knob `ehvi`: "reference" (default) keeps the reference's EHVI / crude 3-D EHVI above; "box" scores
    every 2 to 4 objective problem with the exact EHVI over the box decomposition (`spec_ehvi_box`), built on the
    device or the host as `prep_on_device` selects (`_box_device`); both give the same boxes.

    Additive knob `batch_size` (default 1: one point per iteration, the reference's loop): q > 1 proposes q pool
    rows per iteration by the Kriging believer (`propose_batch`) and evaluates them all; `budget` then counts the
    evaluations after the initial design.

    Additive knob `constrained` (default False: the objectives alone, as above): True optimises a problem with
    inequality constraints (feasible: every constraint <= 0).  One GP per objective and per constraint is fitted, and
    the acquisition is the box EHVI over the front of the feasible samples times the probability that every
    constraint holds (`spec_ehvi_box_feasible`); with no feasible sample yet the front is empty.  It needs
    ehvi="box", no `acquisition_func`, no equality constraints and n_obj + n_ieq_constr <= 8.  The hypervolume
    history counts the feasible samples only (0 while there are none), and `solve` returns a `Constrained_Res` with
    the constraint values in `gsample`."""

    def __init__(self, test_problem, *args, ehvi="reference", batch_size=1, constrained=False, **kwargs):
        if ehvi not in ("reference", "box"):
            raise ValueError(f"ehvi must be 'reference' or 'box' (got {ehvi!r})")
        self.constrained = bool(constrained)
        if self.constrained:
            n_ieq = int(getattr(test_problem, "n_ieq_constr", 0))
            if ehvi != "box":
                raise ValueError("constrained=True scores with the constrained box EHVI: pass ehvi='box'")
            if int(getattr(test_problem, "n_eq_constr", 0)) != 0:
                raise ValueError("constrained=True takes inequality constraints only (the problem has "
                                 f"n_eq_constr={test_problem.n_eq_constr})")
            if n_ieq < 1:
                raise ValueError("constrained=True needs a problem with at least one inequality constraint")
            if test_problem.n_obj + n_ieq > 8:
                raise ValueError(f"constrained=True supports n_obj + n_ieq_constr <= 8 models (got "
                                 f"{test_problem.n_obj} + {n_ieq})")
        super().__init__(test_problem, *args, **kwargs)
        self.ehvi = ehvi
        self.batch_size = self._check_batch_size(batch_size)

    def _get_cached_samples(self, dimensions, sample_exponent):
        return host_prep.cached_samples(dimensions, sample_exponent, seed=int(self.rng.integers(0, 2 ** 31)))

    def solve(self, budget=100, n_init_samples=5, sample_exponent=5, acquisition_func=None):
        if self.constrained:
            if acquisition_func is not None:
                raise ValueError("constrained=True scores with the constrained box EHVI; acquisition_func must be None")
            return self._solve_constrained(budget, n_init_samples)
        if self.batch_size > 1:
            return self._solve_batched(budget, n_init_samples, sample_exponent, acquisition_func)
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
                    spec = spec_ehvi_box(self.max_point, pf, device=self._box_device(pf))
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

    def _batch_spec_for(self, pf, cached_samples, ref_dir=None, acquisition_func=None, min_scalar=None):
        """spec_for(Y_believed) of one batch: the EHVI kinds rebuild the spec from the front of pf and the believed
        rows (max_point fixed for the batch); expected decomposition lowers g_min to the believed rows' minimum.
        A believed row beyond max_point adds no hypervolume and dominates no front point inside it, so it stays out
        of the front (the 2-D stripes need a front inside the reference point)."""
        max_point = np.array(self.max_point, dtype=float)

        def spec_for(Y_bel):
            if acquisition_func is not None:
                g = [acquisition_func(y, ref_dir) for y in Y_bel]
                g_min = float(np.min(np.concatenate([np.ravel(min_scalar), np.ravel(g)])))
                return spec_expected_decomposition(ref_dir, acquisition_func, g_min, cached_samples, self.semantics)
            inside = np.asarray(Y_bel, dtype=float).reshape(-1, self.n_obj)
            inside = inside[np.all(inside <= max_point, axis=1)]
            front = self._calc_pf(np.vstack([pf, inside])) if len(inside) else pf
            if self.ehvi == "box":
                return spec_ehvi_box(max_point, front, device=self._box_device(front))
            if self.n_obj == 2:
                return spec_ehvi(max_point, front, cached_samples, self.semantics)
            return spec_ehvi3d(max_point, front, cached_samples, self.semantics)

        return spec_for

    def _solve_batched(self, budget, n_init_samples, sample_exponent, acquisition_func):
        problem = self.test_problem
        Xsample, ysample = self._initial_design(n_init_samples)
        cached_samples = self._get_cached_samples(self.n_obj, sample_exponent)
        ref_dirs = host_prep.get_reference_directions("das-dennis", self.n_obj, n_partitions=100)
        hypervolume_convergence = []
        done = 0
        while done < budget:
            q = min(self.batch_size, budget - done)
            self._update_bounds(ysample, acquisition_func)
            hypervolume_convergence.append(self._hypervolume(ysample))
            models = self._fit_models(Xsample, [ysample[:, i] for i in range(problem.n_obj)])
            ref_dir = np.asarray(ref_dirs[self.rng.integers(0, len(ref_dirs))])
            min_scalar = None
            if acquisition_func is not None:
                min_scalar = np.min([acquisition_func(y, ref_dir) for y in ysample])
            spec_for = self._batch_spec_for(self._calc_pf(ysample), cached_samples, ref_dir, acquisition_func,
                                            min_scalar)
            X_next, _ = self._propose_batch(models, spec_for, q)
            y_next = np.asarray([self._objective_function(problem, x) for x in X_next]).reshape(q, -1)
            ysample = np.vstack((ysample, y_next))
            Xsample = np.vstack((Xsample, X_next))
            done += q
        mask = self._pareto_members(ysample)
        res = result.Res(ysample[mask], Xsample[mask], ysample, Xsample, hypervolume_convergence, problem.n_obj,
                         n_init_samples)
        res.timings = self.timings
        return res


    def _constrained_spec_for(self, pf):
        """spec_for(Y_believed) of one constrained batch: a believed row (objectives, then constraints) joins the
        feasible front only when every believed constraint is <= 0 and its objectives are inside max_point."""
        max_point = np.array(self.max_point, dtype=float)
        k, c = self.n_obj, self.test_problem.n_ieq_constr

        def spec_for(Y_bel):
            Y = np.asarray(Y_bel, dtype=float).reshape(-1, k + c)
            ok = Y[np.all(Y[:, k:] <= 0, axis=1) & np.all(Y[:, :k] <= max_point, axis=1), :k]
            front = self._calc_pf(np.vstack([pf, ok])) if len(ok) else pf
            return spec_ehvi_box_feasible(max_point, front, c, device=self._box_device(front))

        return spec_for

    def _solve_constrained(self, budget, n_init_samples):
        problem = self.test_problem
        k, c = problem.n_obj, problem.n_ieq_constr
        Xsample, ysample = self._initial_design(n_init_samples)
        gsample = np.asarray([self._constraint_function(problem, x) for x in Xsample]).reshape(-1, c)
        hypervolume_convergence = []
        done = 0
        while done < budget:
            q = min(self.batch_size, budget - done)
            self._update_bounds(ysample)
            y_feasible = ysample[np.all(gsample <= 0, axis=1)]
            hypervolume_convergence.append(self._hypervolume(y_feasible) if len(y_feasible) else 0.0)
            models = self._fit_models(Xsample, [ysample[:, i] for i in range(k)] + [gsample[:, j] for j in range(c)])
            pf = self._calc_pf(y_feasible) if len(y_feasible) else np.empty((0, k))
            if self.batch_size == 1:
                X_next, _ = self._propose(models, spec_ehvi_box_feasible(self.max_point, pf, c,
                                                                         device=self._box_device(pf)))
                X_next = np.atleast_2d(X_next)
            else:
                X_next, _ = self._propose_batch(models, self._constrained_spec_for(pf), q)
            y_next = np.asarray([self._objective_function(problem, x) for x in X_next]).reshape(q, k)
            g_next = np.asarray([self._constraint_function(problem, x) for x in X_next]).reshape(q, c)
            ysample = np.vstack((ysample, y_next))
            Xsample = np.vstack((Xsample, X_next))
            gsample = np.vstack((gsample, g_next))
            done += q
        infeasible = np.any(gsample > 0, axis=1)
        y_feasible, y_infeasible = ysample[~infeasible], ysample[infeasible]
        X_feasible, X_infeasible = Xsample[~infeasible], Xsample[infeasible]
        if len(y_feasible):
            mask = self._pareto_members(y_feasible)
            pf_approx, pf_inputs = y_feasible[mask], X_feasible[mask]
        else:
            pf_approx, pf_inputs = y_feasible, X_feasible
        res = result.Constrained_Res(y_infeasible, y_feasible, X_infeasible, X_feasible, pf_approx, pf_inputs, ysample,
                                     Xsample, hypervolume_convergence, k, n_init_samples)
        res.gsample = gsample
        res.timings = self.timings
        return res


class MonoSurrogateOptimiser(PoolOptimiserBase):
    """One GP on the scalarised objective, closed-form EI (optimisers.py:325-344, :373-527).

    Additive knob `batch_size` (default 1): as for MultiSurrogateOptimiser, q > 1 proposes q points per iteration by
    the Kriging believer and `budget` counts evaluations after the initial design."""

    def __init__(self, test_problem, *args, batch_size=1, **kwargs):
        super().__init__(test_problem, *args, **kwargs)
        self.batch_size = self._check_batch_size(batch_size)

    @staticmethod
    def _batch_spec_for(current_best):
        """spec_for(Y_believed) of one batch: EI against the minimum of the incumbent and the believed values."""
        def spec_for(Y_bel):
            best = min(float(current_best), float(np.min(Y_bel))) if len(Y_bel) else float(current_best)
            return spec_ei(best, 0.0)

        return spec_for

    def _normalize_data(self, data):
        return (data - np.min(data)) / (np.max(data) - np.min(data))

    def solve(self, aggregation_func, budget=100, n_init_samples=5):
        if self.batch_size > 1:
            return self._solve_batched(aggregation_func, budget, n_init_samples)
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

    def _solve_batched(self, aggregation_func, budget, n_init_samples):
        problem = self.test_problem
        weights = np.asarray([1 / problem.n_obj] * problem.n_obj)
        Xsample, ysample = self._initial_design(n_init_samples)
        self._update_bounds(ysample, aggregation_func)
        aggregated_samples = np.asarray([aggregation_func(y, weights) for y in ysample]).flatten()
        ref_dirs = host_prep.get_reference_directions("das-dennis", problem.n_obj, n_partitions=100)
        hypervolume_convergence = []
        done = 0
        while done < budget:
            q = min(self.batch_size, budget - done)
            self._update_bounds(ysample, aggregation_func)
            hypervolume_convergence.append(self._hypervolume(ysample))
            current_best = aggregated_samples[np.argmin(aggregated_samples)]
            model = self._fit_model(Xsample, aggregated_samples)
            next_X, _ = self._propose_batch([model], self._batch_spec_for(current_best), q)
            for x in next_X:
                next_y = self._objective_function(problem, x)
                ysample = np.vstack((ysample, next_y))
                ref_dir = ref_dirs[self.rng.integers(0, len(ref_dirs))]
                aggregated_samples = np.append(aggregated_samples, aggregation_func(next_y, ref_dir))
            Xsample = np.vstack((Xsample, next_X))
            done += q
        mask = self._pareto_members(ysample)
        res = result.Res(ysample[mask], Xsample[mask], ysample, Xsample, hypervolume_convergence, problem.n_obj,
                         n_init_samples)
        res.timings = self.timings
        return res
