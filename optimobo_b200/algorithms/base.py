"""Shared outer-loop plumbing of the re-hosted optimisers.

The BO outer loops (LHS init -> per iteration: bounds, hypervolume, GP fit, acquisition,
evaluate, append) are host orchestration and are out of scope for kernels (SURVEY.md section 2,
rows 3-7); they are re-hosted thinly so `.solve()` keeps working.  What changes is the seam
`_get_proposed*`: where the reference calls `scipy.optimize.differential_evolution(obj, bounds)`
(optimisers.py:87,118,366; cparego.py:94,544; emo.py:240) or a 20-member / 1000-generation EA
(parego.py:242-270, keep.py:260-292) that evaluates the acquisition one x at a time, this path
scores a pool of `n_candidates` points in one fused GPU pass and takes the arg-max.

Additive knobs (reference defaults untouched): n_candidates, precision {"auto","fp64","fast"},
semantics {"reference","exact"}, device, seed, fit (callable or fixed hyper-parameters).
"""
from __future__ import annotations

import time

import numpy as np
import torch

from .. import device_prep, host_prep
from ..acquisition import CandidatePool, propose, propose_batch
from ..fit import fit_hyperparameters, fit_hyperparameters_device
from ..gp import GPModel

# "auto" builds the box decomposition on the device from this front size on: on the B200 the device is faster at every
# front size measured, and from 16 points the host takes 4.6x (k = 3) to 24x (k = 4) its time (DESIGN.md section 4)
BOX_DEVICE_MIN_FRONT = 16
BOX_DEVICE_MAX_FRONT = 512      # ombo_ehvi_boxes takes fronts of up to 512 distinct points


class PoolOptimiserBase:
    def __init__(self, test_problem, ideal_point=None, max_point=None, n_candidates=1 << 16, precision="auto",
                 semantics="reference", device="cuda:0", seed=None, hyperparameters=None, max_f_eval=1000,
                 fit_on_device=True, refine_rounds=2, prep_on_device="auto"):
        self.test_problem = test_problem
        self.max_point = max_point
        self.ideal_point = ideal_point
        self.n_vars = test_problem.n_var
        self.n_obj = test_problem.n_obj
        self.upper = test_problem.xu
        self.lower = test_problem.xl
        self.is_ideal_known = ideal_point is not None
        self.is_max_known = max_point is not None
        # --- B200-path knobs ---
        self.n_candidates = int(n_candidates)
        self.precision = precision
        self.semantics = semantics
        self.device = device
        self.rng = np.random.default_rng(seed)
        self.hyperparameters = hyperparameters      # (lengthscale, variance) to skip the fit (parity tests)
        self.max_f_eval = max_f_eval
        self.fit_on_device = fit_on_device       # likelihood + gradient on the GPU (ombo_gp_nlml_grad)
        self.refine_rounds = refine_rounds       # zoom rounds around the pool winner (DE's polish step)
        # first front / hypervolume / cells on the device (bit-identical to host_prep; "auto": once the sample
        # holds >= 512 rows, where the O(n^2) host versions start to show next to a ~100 ms scoring pass); the box
        # decomposition (box EHVI, EMO for 3 and 4 objectives) follows its own rule (_box_device)
        self.prep_on_device = prep_on_device
        self.timings = []

    # ---- problem access ------------------------------------------------------------------------
    def _objective_function(self, problem, x):
        return problem.evaluate(x)

    def _constraint_function(self, problem, x):
        return problem.evaluate_constraints(x)

    def _initial_design(self, n_init_samples):
        ranges = list(zip(self.test_problem.xl, self.test_problem.xu))
        X = host_prep.latin_hypercube(n_init_samples, ranges, self.rng)
        Y = np.asarray([self._objective_function(self.test_problem, x) for x in X])
        return X, Y

    # ---- bounds bookkeeping (optimisers.py:190-213 and its copies) ---------------------------
    def _update_bounds(self, ysample, scalarisation=None):
        changed = False
        if not self.is_max_known:
            self.max_point = ysample.max(axis=0)
            changed = True
        if not self.is_ideal_known:
            self.ideal_point = ysample.min(axis=0)
            changed = True
        if changed and scalarisation is not None:
            scalarisation.set_bounds(self.ideal_point, self.max_point)

    def _prep_device(self, rows):
        return self.prep_on_device is True or (self.prep_on_device == "auto" and rows >= 512)

    def _hypervolume(self, ysample, ref_point=None):
        ref = self.max_point if ref_point is None else ref_point
        if self._prep_device(len(ysample)) and np.shape(ysample)[1] in (2, 3):
            return device_prep.hypervolume(ysample, ref, self.device)
        return host_prep.hypervolume(ysample, ref)

    def _calc_pf(self, ysample):
        if self._prep_device(len(ysample)):
            return device_prep.calc_pf(ysample, self.device)
        return host_prep.calc_pf(ysample)

    def _box_device(self, front):
        """Where the box decomposition of `front` is built: self.device when prep_on_device is True (or "auto" and the
        front has at least BOX_DEVICE_MIN_FRONT rows) and the front is finite and within the device limit, else None
        (the host)."""
        front = np.asarray(front, dtype=float)
        n = len(front)
        if self.prep_on_device is True:
            wanted = True
        elif self.prep_on_device == "auto":
            wanted = n >= BOX_DEVICE_MIN_FRONT
        else:
            wanted = False
        ok = n <= BOX_DEVICE_MAX_FRONT and bool(np.all(np.isfinite(front)))
        return self.device if wanted and ok else None

    # ---- surrogate ---------------------------------------------------------------------------------
    def _fit_model(self, X, y):
        t0 = time.perf_counter()
        if self.hyperparameters is not None:
            ell, sf2 = self.hyperparameters
        else:
            fit = fit_hyperparameters_device if self.fit_on_device else fit_hyperparameters
            kw = dict(device=self.device) if self.fit_on_device else {}
            ell, sf2 = fit(X, y, max_f_eval=self.max_f_eval, **kw)
        t1 = time.perf_counter()
        model = GPModel(X, y, ell, sf2, noise=0.0, device=self.device)
        self._t_fit = getattr(self, "_t_fit", 0.0) + (t1 - t0)
        self._t_refresh = getattr(self, "_t_refresh", 0.0) + (time.perf_counter() - t1)
        return model

    def _fit_models(self, X, columns):
        """One surrogate per column of `columns` (objectives / constraints), fitted and refreshed CONCURRENTLY: a fit
        is a chain of small dependent launches (K3 per likelihood evaluation) that leaves the GPU mostly idle, so the
        models' chains overlap on separate streams, one host thread each (see gp.refresh_models)."""
        cols = [np.asarray(c) for c in columns]
        if len(cols) <= 1 or not torch.cuda.is_available():
            return [self._fit_model(X, c) for c in cols]
        from concurrent.futures import ThreadPoolExecutor
        dev = torch.device(self.device) if self.device is not None else torch.device("cuda", torch.cuda.current_device())
        cur = torch.cuda.current_stream(dev)
        streams = [torch.cuda.Stream(dev) for _ in cols]
        for st in streams:
            st.wait_stream(cur)

        def work(arg):
            c, st = arg
            with torch.cuda.device(dev), torch.cuda.stream(st):
                return self._fit_model(X, c)

        with ThreadPoolExecutor(len(cols)) as ex:
            models = list(ex.map(work, zip(cols, streams)))
        for st in streams:
            cur.wait_stream(st)
        return models

    def _precision_for(self, models):
        from ..acquisition import resolve_precision
        return resolve_precision(models, self.precision)

    # ---- the seam: pool scoring + arg-max instead of DE / EA ---------------------------------
    def _propose(self, models, spec):
        t0 = time.perf_counter()
        pool = CandidatePool.counter(self.n_candidates, self.test_problem.xl, self.test_problem.xu,
                                     seed=int(self.rng.integers(1, 2 ** 62)))
        x, neg_value, index = propose(models, spec, pool, precision=self._precision_for(models),
                                      refine_rounds=self.refine_rounds)
        self.timings.append(dict(fit_s=getattr(self, "_t_fit", 0.0), refresh_s=getattr(self, "_t_refresh", 0.0),
                                 score_s=time.perf_counter() - t0, n_candidates=self.n_candidates))
        self._t_fit = self._t_refresh = 0.0
        return x, neg_value

    def _propose_batch(self, models, spec_for, q):
        """q pool rows by the Kriging believer (acquisition.propose_batch); one timing record for the batch."""
        t0 = time.perf_counter()
        pool = CandidatePool.counter(self.n_candidates, self.test_problem.xl, self.test_problem.xu,
                                     seed=int(self.rng.integers(1, 2 ** 62)))
        X, neg_values, _, certified = propose_batch(models, spec_for, pool, q, precision=self._precision_for(models))
        self.timings.append(dict(fit_s=getattr(self, "_t_fit", 0.0), refresh_s=getattr(self, "_t_refresh", 0.0),
                                 score_s=time.perf_counter() - t0, n_candidates=self.n_candidates, batch=q,
                                 certified=int(certified.sum())))
        self._t_fit = self._t_refresh = 0.0
        return X, neg_values

    @staticmethod
    def _check_batch_size(batch_size):
        if int(batch_size) != batch_size or batch_size < 1:
            raise ValueError(f"batch_size must be a positive integer (got {batch_size!r})")
        return int(batch_size)

    # ---- result ------------------------------------------------------------------------------------
    @staticmethod
    def _pareto_members(ysample):
        if len(ysample) <= 1:
            return np.ones(len(ysample), bool)
        mask = host_prep.pareto_mask(ysample)
        return mask
