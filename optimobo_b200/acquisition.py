"""Batched acquisition evaluation + arg-max over candidate pools: the drop-in for the
reference's per-candidate acquisition callables and the inner optimiser that calls them.

Reference seam (SURVEY.md section 8b):
    function(X, models, max_point, pf, cache)                 EHVI / EHVI_3D   optimisers.py:112
    function(X, models, ref_dir, scalar_func, min_val, cache) expected_decomposition   :84
    function(X, model, current_best)                          _expected_improvement    :362
    function(X, agg_model, constraint_models, current_best)   consraint_ei     cparego.py:540
    function(X, models, P, cells)                             hypervolume_based_PoI  emo.py:237
    function(X, models, ideal_point, max_point, PF)           hypervolume_based_PoI_box (2 to 4 objectives)
each called with ONE x by scipy differential_evolution or the ParEGO/KEEP EA.  Here the same
names accept X of shape (d,) or (m, d) and return (m,) values computed on the GPU, and
`propose*` scores a whole pool (explicit or counter-generated) and returns
`(x_best, -acq_best)` like `(res.x, res.fun)`.

Everything goes through the C ABI (`_cabi`); there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import warnings
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _cabi, host_prep
from .gp import GPModel, _as_device, current_stream_ptr

_PREC = {"fp64": _cabi.PREC_FP64, "fast": _cabi.PREC_FAST}


def resolve_precision(models, precision):
    """'fp64' | 'fast' | 'auto' -> 'fp64' | 'fast'.  'auto' picks the fast mode exactly where its accuracy is
    guaranteed: the tcgen05 path is built, n >= 64 (tiny GPs are cheap in FP64), d <= 24 and the conditioning
    proxy of EVERY model is below GPModel.FAST_MODE_CONDITIONING_LIMIT (scripts/cond_study.py); many points per
    length-scale in few dimensions (README MyProblem: kappa ~ 1e8) run FP64.  An explicit 'fast' on an
    ill-conditioned GP is honoured with a RuntimeWarning."""
    models = [models] if isinstance(models, GPModel) else list(models)
    if precision == "auto":
        n = max(m.n for m in models)
        if not (_cabi.fast_path_available() and n >= 64 and models[0].d <= 24):
            return "fp64"
        return "fast" if max(m.conditioning for m in models) <= GPModel.FAST_MODE_CONDITIONING_LIMIT else "fp64"
    if precision not in _PREC:
        raise ValueError(f"precision must be 'fp64', 'fast' or 'auto' (got {precision!r})")
    if precision == "fast":
        worst = max(m.conditioning for m in models)
        if worst > GPModel.FAST_MODE_CONDITIONING_LIMIT:
            warnings.warn(f"fast precision on an ill-conditioned GP (conditioning proxy {worst:.1e} > "
                          f"{GPModel.FAST_MODE_CONDITIONING_LIMIT:.0e}): sigma may be off by more than 1e-3 sigma_f; "
                          "use precision='fp64' or 'auto'", RuntimeWarning, stacklevel=3)
    return precision
_SEM = {"reference": _cabi.SEM_REFERENCE, "exact": _cabi.SEM_EXACT}


# --------------------------------------------------------------------------------------------
# candidate pools
# --------------------------------------------------------------------------------------------
@dataclass
class CandidatePool:
    """Either an explicit (m, d) CUDA tensor (float64 / float32) or a counter-generated uniform
    pool over the box [lo, hi): row i, column j = lo_j + (hi_j - lo_j) * u(seed, i*d + j).  The
    generated pool is never materialised; any shard (index_base, m) of it is reproducible on
    any GPU."""
    m: int
    d: int
    X: torch.Tensor | None = None
    lo: np.ndarray | None = None
    hi: np.ndarray | None = None
    seed: int = 1
    index_base: int = 0

    @classmethod
    def explicit(cls, X, device=None, index_base=0):
        if not torch.is_tensor(X):
            X = torch.as_tensor(np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64))))
        if X.dtype not in (torch.float64, torch.float32):
            X = X.double()
        if device is not None:
            X = X.to(device)
        if not X.is_cuda:
            raise RuntimeError("explicit candidate pools must live on the GPU (use propose_host for host buffers)")
        X = X.contiguous()
        return cls(m=X.shape[0], d=X.shape[1], X=X, index_base=index_base)

    @classmethod
    def counter(cls, m, lo, hi, seed=1, index_base=0):
        lo = np.asarray(lo, dtype=np.float64).reshape(-1)
        hi = np.asarray(hi, dtype=np.float64).reshape(-1)
        return cls(m=int(m), d=len(lo), lo=lo, hi=hi, seed=int(seed), index_base=int(index_base))

    def shard(self, rank, world):
        """Contiguous slice of the global index range for `rank` of `world` (SURVEY section 8e)."""
        per = (self.m + world - 1) // world
        start = min(rank * per, self.m)
        stop = min(start + per, self.m)
        if self.X is not None:
            return CandidatePool(m=stop - start, d=self.d, X=self.X[start:stop], index_base=self.index_base + start)
        return CandidatePool(m=stop - start, d=self.d, lo=self.lo, hi=self.hi, seed=self.seed,
                             index_base=self.index_base + start)

    def c_struct(self, host_ptr=None, host_dtype=None):
        p = _cabi.Pool()
        p.m, p.d, p.index_base, p.seed = self.m, self.d, self.index_base, self.seed
        if host_ptr is not None:
            p.X, p.dtype = host_ptr, host_dtype
        elif self.X is not None:
            p.X = self.X.data_ptr()
            p.dtype = 0 if self.X.dtype == torch.float64 else 1
        else:
            p.X, p.dtype = None, 0
            for j in range(self.d):
                p.lo[j], p.hi[j] = self.lo[j], self.hi[j]
        return p

    def rows(self, index, count=1, device=None):
        """Rows [index, index+count) (global indices) as a (count, d) float64 CUDA tensor."""
        if self.X is not None:
            i = index - self.index_base
            return self.X[i:i + count].double()
        dev = _as_device(device)
        out = torch.empty((count, self.d), dtype=torch.float64, device=dev)
        ctx = _cabi.Context.get(dev.index)
        p = self.c_struct()
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib().ombo_pool_rows(ctx.handle, C.byref(p), index, count,
                                                   C.c_void_p(out.data_ptr()), current_stream_ptr(dev)))
        return out


# --------------------------------------------------------------------------------------------
# acquisition specifications
# --------------------------------------------------------------------------------------------
@dataclass
class AcquisitionSpec:
    kind: int
    semantics: str = "reference"
    n_obj: int = 0
    best: float = 0.0
    var_eps: tuple = ()
    ref: tuple = ()
    ideal: tuple = ()
    maxp: tuple = ()
    weights: tuple = ()
    scalarisation: int = 0
    sc_params: tuple = (0.0, 0.0, 0.0, 0.0)
    cache_c: tuple = (0.0, 0.0)
    stripes: np.ndarray | None = None
    cells: np.ndarray | None = None
    cache: np.ndarray | None = None
    n_models: int = 1
    reserved: int = 0          # ombo_acq.reserved (EHVI2D: _cabi.ACQ_FRONT_VALID)
    _dev: dict = field(default_factory=dict, repr=False)

    def c_struct(self, device):
        a = _cabi.Acq()
        a.kind, a.semantics, a.scalarisation, a.n_obj = self.kind, _SEM[self.semantics], self.scalarisation, self.n_obj
        a.best = float(self.best)
        for dst, src in ((a.var_eps, self.var_eps), (a.ref, self.ref), (a.ideal, self.ideal),
                         (a.maxp, self.maxp), (a.weights, self.weights), (a.sc_params, self.sc_params)):
            for i, v in enumerate(src):
                dst[i] = float(v)
        a.cache_c00, a.cache_c01 = self.cache_c
        a.reserved = self.reserved

        def up(name, arr):
            if (torch.is_tensor(arr) and arr.device == torch.device(device) and arr.dtype == torch.float64
                    and arr.is_contiguous()):
                return arr.data_ptr()                   # already where the kernels read it: no copy
            key = (name, str(device))
            if key not in self._dev:
                self._dev[key] = (arr.to(device=device, dtype=torch.float64).contiguous() if torch.is_tensor(arr) else
                                  torch.as_tensor(np.ascontiguousarray(arr, dtype=np.float64)).to(device))
            return self._dev[key].data_ptr()

        if self.stripes is not None:
            a.stripes = up("stripes", self.stripes)
            # EHVI2D: stripes are (2, P + 2); EHVI_BOX(_FEAS), HV_POI_BOX: the (k, B) breakpoint table
            box = self.kind in (_cabi.ACQ_EHVI_BOX, _cabi.ACQ_EHVI_BOX_FEAS, _cabi.ACQ_HV_POI_BOX)
            a.n_pf = self.stripes.shape[1] - (0 if box else 2)
        if self.cells is not None:
            a.cells = up("cells", self.cells)
            a.n_cells = self.cells.shape[0]
        if self.cache is not None:
            a.cache = up("cache", self.cache)
            a.n_samples = self.cache.shape[0]
        return a


def spec_ehvi(max_point, PF, cache, semantics="reference"):
    """util_functions.py:136-167."""
    PF = np.atleast_2d(np.asarray(PF, dtype=np.float64))
    if PF.shape[1] != 2:
        raise ValueError("EHVI is 2-objective; use spec_ehvi3d for 3 objectives")
    valid = host_prep.front_is_staircase(PF, max_point)
    return AcquisitionSpec(kind=_cabi.ACQ_EHVI2D, semantics=semantics, n_obj=2, ref=tuple(max_point),
                           stripes=host_prep.ehvi_stripes(PF, max_point),
                           cache_c=host_prep.cache_covariance(cache), n_models=2,
                           reserved=_cabi.ACQ_FRONT_VALID if valid else 0)


def spec_ehvi3d(max_point, PF, cache, semantics="reference"):
    """util_functions.py:170-214; Sminus = HV(PF) is hoisted to the host."""
    cache = np.asarray(cache, dtype=np.float64)
    k = cache.shape[1]
    return AcquisitionSpec(kind=_cabi.ACQ_EHVI3D, semantics=semantics, n_obj=k, ref=tuple(max_point),
                           best=host_prep.hypervolume(PF, max_point), cache=cache, n_models=k)


def _box_tables(PF, r, device):
    """(table, boxes as float64) of the box decomposition: host_prep.ehvi_boxes as numpy arrays, or with a device its
    device twin (device_prep.ehvi_boxes, equal element for element) as tensors on that device."""
    if device is not None:
        from . import device_prep
        return device_prep.ehvi_boxes(PF, r, device)
    table, boxes = host_prep.ehvi_boxes(PF, r)
    return table, boxes.astype(np.float64)


def spec_ehvi_box(max_point, PF, device=None):
    """Exact expected hypervolume improvement for 2 <= k <= 4 objectives: sum over the disjoint boxes of the region
    no front point dominates (host_prep.ehvi_boxes) of prod_i (H_i(u_i) - H_i(l_i)), H_i(t) = E[(t - y_i)^+], with each
    model's own mean and variance.  Not a reference acquisition; `semantics` does not apply.  With `device`, the
    decomposition is built there (device_prep.ehvi_boxes) and the spec holds its device tensors."""
    r = np.asarray(max_point, dtype=np.float64).reshape(-1)
    table, boxes = _box_tables(PF, r, device)
    k = len(r)
    return AcquisitionSpec(kind=_cabi.ACQ_EHVI_BOX, n_obj=k, ref=tuple(r), stripes=table, cells=boxes, n_models=k)


def spec_ehvi_box_feasible(max_point, PF, n_constraints, var_eps=1e-5, device=None):
    """Constrained box EHVI: spec_ehvi_box(max_point, PF) times the probability that every constraint holds,
    prod_j Phi(-mu_j / sqrt(var_j + var_eps)), with models = k objective GPs followed by `n_constraints` constraint GPs
    (feasible: every constraint <= 0).  PF is the front of the feasible samples; an empty front scores against the
    single box [-inf, r].  var_eps defaults to the 1e-5 of the constrained EI's feasibility factor (cparego.py:486-496);
    0 is allowed.  Not a reference acquisition; `semantics` does not apply.  `device` as for spec_ehvi_box."""
    r = np.asarray(max_point, dtype=np.float64).reshape(-1)
    k, c = len(r), int(n_constraints)
    if c != n_constraints or not 1 <= c <= _cabi.MAX_GP - k:
        raise ValueError(f"n_constraints must be an integer in 1..{_cabi.MAX_GP - k} for {k} objectives "
                         f"(got {n_constraints!r})")
    if not var_eps >= 0:
        raise ValueError(f"var_eps must be >= 0 (got {var_eps!r})")
    table, boxes = _box_tables(np.asarray(PF, dtype=np.float64).reshape(-1, k), r, device)
    return AcquisitionSpec(kind=_cabi.ACQ_EHVI_BOX_FEAS, n_obj=k, ref=tuple(r), stripes=table,
                           cells=boxes, var_eps=(0.0,) * k + (float(var_eps),) * c,
                           n_models=k + c)


def spec_expected_decomposition(weights, agg_func, agg_function_min, cache, semantics="reference"):
    """util_functions.py:285-327.  `agg_func` is a live scalarisation object; its bounds are read
    now (they mutate every BO iteration)."""
    cache = np.asarray(cache, dtype=np.float64)
    k = cache.shape[1]
    if not hasattr(agg_func, "device_spec"):
        agg_func = adopt_scalarisation(agg_func)
    sc_id, params = agg_func.device_spec()
    return AcquisitionSpec(kind=_cabi.ACQ_EXPECTED_DECOMP, semantics=semantics, n_obj=k,
                           best=float(np.asarray(agg_function_min).reshape(-1)[0]),
                           ideal=tuple(np.asarray(agg_func.ideal_point, float)),
                           maxp=tuple(np.asarray(agg_func.max_point, float)),
                           weights=tuple(np.asarray(weights, float).reshape(-1)),
                           scalarisation=sc_id, sc_params=params, cache=cache, n_models=k)


def spec_ei(current_best, var_eps=0.0):
    """optimisers.py:325-344 / cparego.py:450-469 (var_eps=0); parego.py:126-145 / keep.py:118-137 (1e-6)."""
    return AcquisitionSpec(kind=_cabi.ACQ_EI, best=float(current_best), var_eps=(var_eps,), n_models=1)


def spec_constrained_ei(current_best, n_constraints):
    """cparego.py:486-496: EI(agg) * prod_c Phi((0 - mu_c)/sqrt(var_c + 1e-5))."""
    return AcquisitionSpec(kind=_cabi.ACQ_CONSTRAINED_EI, best=float(current_best),
                           var_eps=(0.0,) + (1e-5,) * n_constraints, n_models=1 + n_constraints)


def spec_pareto_ei(current_best):
    """keep.py:142-150: models = [pareto_model, scalarised_model]."""
    return AcquisitionSpec(kind=_cabi.ACQ_PARETO_EI, best=float(current_best), var_eps=(0.0, 1e-6), n_models=2)


def spec_hv_poi(cells):
    """emo.py:192-228: cells (n_cells, 2, 2), [c][0] upper / [c][1] lower."""
    cells = np.asarray(cells, dtype=np.float64)
    return AcquisitionSpec(kind=_cabi.ACQ_HV_POI, n_obj=2, var_eps=(1e-5, 1e-5), cells=cells, n_models=2)


def spec_hv_poi_box(ideal_point, max_point, PF, device=None):
    """The hypervolume-based probability of improvement of spec_hv_poi (emo.py:192-228) for 2 <= k <= 4 objectives:
    PoI * Imp over the region R = {ideal <= z <= r' : no front point dominates z}, r' = max(max_point, PF.max(0)) per
    objective, with PoI = P(y in R) and Imp = vol(R above mu) at sigma_i = sqrt(var_i + 1e-5).  Both depend on R only;
    for k = 2, R is the region decompose_into_cells tiles, so the value equals spec_hv_poi's on those cells whenever
    no front point lies below the ideal point.  R is tiled by the boxes of ehvi_boxes(PF, r') with every breakpoint
    clamped below at the ideal point; an empty front gives the single box [ideal, max_point].  `device` as for
    spec_ehvi_box."""
    ideal = np.asarray(ideal_point, dtype=np.float64).reshape(-1)
    maxp = np.asarray(max_point, dtype=np.float64).reshape(-1)
    k = len(maxp)
    if not 2 <= k <= 4 or len(ideal) != k:
        raise ValueError(f"HV-PoI over boxes takes 2 to 4 objectives and an ideal point of the same length "
                         f"(got {len(ideal)} and {k})")
    P = np.asarray(PF.detach().cpu() if torch.is_tensor(PF) else PF, dtype=np.float64).reshape(-1, k)
    if not (np.all(np.isfinite(ideal)) and np.all(np.isfinite(maxp)) and np.all(np.isfinite(P))):
        raise ValueError("HV-PoI over boxes needs a finite ideal point, max point and front")
    r = np.maximum(maxp, P.max(0)) if len(P) else maxp
    table, boxes = _box_tables(P, r, device)
    if torch.is_tensor(table):
        table = torch.maximum(table, torch.as_tensor(ideal, device=table.device)[:, None])
    else:
        table = np.maximum(table, ideal[:, None])
    return AcquisitionSpec(kind=_cabi.ACQ_HV_POI_BOX, n_obj=k, ref=tuple(r), var_eps=(1e-5,) * k, stripes=table,
                           cells=boxes, n_models=k)


def adopt_scalarisation(obj):
    """Maps a *reference* `optimobo.scalarisations` object (duck-typed by class name and live
    attributes) onto this package's class so the CUDA switch can serve it."""
    from . import scalarisations as S
    cls = getattr(S, type(obj).__name__, None)
    if cls is None or not issubclass(cls, S.Scalarisation):
        raise TypeError(f"no CUDA implementation for scalarisation {type(obj).__name__!r} (no CPU fallback)")
    new = cls.__new__(cls)
    new.__dict__.update(vars(obj))
    return new


# --------------------------------------------------------------------------------------------
# scoring
# --------------------------------------------------------------------------------------------
@dataclass
class ScoreResult:
    mu: torch.Tensor | None
    var: torch.Tensor | None
    acq: torch.Tensor | None
    best_value: float | None
    best_index: int | None
    best_dev: torch.Tensor | None = None


def _models_list(models):
    return [models] if isinstance(models, GPModel) else list(models)


def _checked_models(models, pool):
    models = _models_list(models)
    dev = models[0].device
    for mdl in models:
        if not isinstance(mdl, GPModel):
            raise TypeError("models must be optimobo_b200.GPModel instances (GPModel.from_gpy adopts GPy models)")
        if mdl.device != dev:
            raise ValueError("all models must live on the same device")
    if pool.X is not None and pool.X.device != dev:
        raise ValueError("pool and models are on different devices")
    return models, dev


def score(models, spec, pool, precision="fp64", want_posterior=False, want_acq=False, want_best=True,
          var_floor=1e-15, sync=True):
    """One pass of the hot path over `pool` (K1+K2 per model, K4, K5)."""
    models, dev = _checked_models(models, pool)
    precision = resolve_precision(models, precision)
    G = len(models)
    gps = (_cabi.Gp * G)(*[m.c_struct(var_floor) for m in models])
    p = pool.c_struct()
    if spec is None:
        a = _cabi.Acq()
        a.kind = _cabi.ACQ_NONE
        want_best = False
    else:
        if spec.n_models > G:
            raise ValueError(f"acquisition needs {spec.n_models} models, got {G}")
        a = spec.c_struct(dev)
    mu = var = acq = best = None
    if want_posterior:
        mu = torch.empty((G, pool.m), dtype=torch.float64, device=dev)
        var = torch.empty((G, pool.m), dtype=torch.float64, device=dev)
    if want_acq:
        acq = torch.empty((pool.m,), dtype=torch.float64, device=dev)
    if want_best:
        best = torch.empty((2,), dtype=torch.int64, device=dev)
    ctx = _cabi.Context.get(dev.index)
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_score(ctx.handle, gps, G, C.byref(p), C.byref(a), _PREC[precision],
                                           ptr(mu), ptr(var), ptr(acq), ptr(best), current_stream_ptr(dev)))
    bv = bi = None
    if want_best and sync:
        host = best.cpu()
        bv = float(host[:1].view(torch.float64)[0])
        bi = int(host[1])
    return ScoreResult(mu, var, acq, bv, bi, best)


def acquire_from_posterior(spec, mu, var, device="cuda:0", index_base=0):
    """K4+K5 on caller-supplied posteriors mu/var (n_models, m): returns (acq (m,) CUDA tensor,
    best_value, best_index)."""
    dev = _as_device(device)
    mu_t = torch.as_tensor(np.ascontiguousarray(np.atleast_2d(np.asarray(mu, dtype=np.float64)))).to(dev)
    var_t = torch.as_tensor(np.ascontiguousarray(np.atleast_2d(np.asarray(var, dtype=np.float64)))).to(dev)
    G, m = mu_t.shape
    a = spec.c_struct(dev)
    acq = torch.empty((m,), dtype=torch.float64, device=dev)
    best = torch.empty((2,), dtype=torch.int64, device=dev)
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_acquire_posterior(
            ctx.handle, C.byref(a), G, C.c_void_p(mu_t.data_ptr()), C.c_void_p(var_t.data_ptr()), m, m,
            index_base, C.c_void_p(acq.data_ptr()), C.c_void_p(best.data_ptr()), current_stream_ptr(dev)))
    host = best.cpu()
    return acq, float(host[:1].view(torch.float64)[0]), int(host[1])


def scalarise_on_device(agg_func, F, weights, device="cuda:0"):
    """g(F[r, :], weights) for every row of F (m, k) through the CUDA scalarisation switch -- the device twin of
    `agg_func(F, weights)` (scalarisations.py:20-27).  `agg_func` is a scalarisation object of this package or of
    the reference (adopted by class name); returns a (m,) numpy array."""
    dev = _as_device(device)
    if not hasattr(agg_func, "device_spec"):
        agg_func = adopt_scalarisation(agg_func)
    Fh = np.ascontiguousarray(np.atleast_2d(np.asarray(F, dtype=np.float64)))
    m, k = Fh.shape
    if k > _cabi.MAX_OBJ:
        raise ValueError(f"the device scalarisation switch takes up to {_cabi.MAX_OBJ} objectives (got {k})")
    sc_id, params = agg_func.device_spec()
    spec = AcquisitionSpec(kind=_cabi.ACQ_EXPECTED_DECOMP, n_obj=k, scalarisation=sc_id, sc_params=params,
                           ideal=tuple(np.asarray(agg_func.ideal_point, float)),
                           maxp=tuple(np.asarray(agg_func.max_point, float)),
                           weights=tuple(np.asarray(weights, float).reshape(-1)))
    a = spec.c_struct(dev)
    Fd = torch.as_tensor(Fh).to(dev)
    out = torch.empty((m,), dtype=torch.float64, device=dev)
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_scalarise(ctx.handle, C.byref(a), C.c_void_p(Fd.data_ptr()), m,
                                               C.c_void_p(out.data_ptr()), current_stream_ptr(dev)))
    return out.cpu().numpy()


def posterior(models, X, precision="fp64", var_floor=1e-15):
    """(mu, var), each (n_models, m) float64 CUDA tensors, for explicit candidates X."""
    models = _models_list(models)
    pool = X if isinstance(X, CandidatePool) else CandidatePool.explicit(X, device=models[0].device)
    r = score(models, None, pool, precision=precision, want_posterior=True, var_floor=var_floor)
    return r.mu, r.var


def evaluate(models, spec, X, precision="fp64"):
    """Acquisition values (m,) as a numpy array for explicit candidates X ((d,) or (m,d))."""
    models = _models_list(models)
    Xa = np.atleast_2d(np.asarray(X.detach().cpu() if torch.is_tensor(X) else X, dtype=np.float64))
    pool = CandidatePool.explicit(Xa, device=models[0].device)
    r = score(models, spec, pool, precision=precision, want_acq=True, want_best=False)
    return r.acq.cpu().numpy()


def polish(models, spec, starts, lo, hi, max_iter=30, fd_step=1e-5, precision="fp64"):
    """SURVEY section 8f rank 3: local refinement of the best pool candidates, mirroring the `polish=True` step of
    scipy's differential_evolution that every inner-optimiser call site of the reference runs after its global phase
    (optimisers.py:87,118,366; cparego.py:94,544; emo.py:240 -- scipy polishes with
    `minimize(fun, x, method="L-BFGS-B", bounds=...)` and finite-difference gradients).

    `starts` (k, d): every start is polished by its own bounded L-BFGS-B run on the host; ALL acquisition evaluations
    go through the GPU scoring kernels -- the objective value and the 2 d central-difference points of a gradient are
    ONE batched scoring call of 2 d + 1 candidates (FP64 mode: finite differences need the smooth arithmetic).
    Returns (x_best (d,), acq_best, per-start acquisition values (k,))."""
    from scipy.optimize import minimize
    models = _models_list(models)
    lo = np.asarray(lo, dtype=np.float64)
    hi = np.asarray(hi, dtype=np.float64)
    starts = np.atleast_2d(np.asarray(starts, dtype=np.float64))
    d = starts.shape[1]
    h = fd_step * (hi - lo)

    def fun_and_grad(x):
        # forward / backward points clipped to the box; one GPU call for value + gradient
        xp = np.minimum(x + h, hi)
        xm = np.maximum(x - h, lo)
        batch = np.vstack([x[None, :], np.where(np.eye(d, dtype=bool), xp[None, :], x[None, :]),
                           np.where(np.eye(d, dtype=bool), xm[None, :], x[None, :])])
        v = evaluate(models, spec, batch, precision=precision)
        v = np.where(np.isfinite(v), v, -1e300)
        g = (v[1:d + 1] - v[d + 1:]) / np.maximum(xp - xm, 1e-300)
        return -v[0], -g

    best_x, best_v, vals = None, -np.inf, []
    for x0 in starts:
        res = minimize(fun_and_grad, np.clip(x0, lo, hi), jac=True, method="L-BFGS-B", bounds=list(zip(lo, hi)),
                       options=dict(maxiter=max_iter))
        v = float(evaluate(models, spec, res.x[None, :], precision=precision)[0])
        v0 = float(evaluate(models, spec, np.clip(x0, lo, hi)[None, :], precision=precision)[0])
        xk, vk = (res.x, v) if (np.isfinite(v) and v >= v0) else (np.clip(x0, lo, hi), v0)    # never worse than the start
        vals.append(vk)
        if vk > best_v:
            best_x, best_v = xk, vk
    return best_x, best_v, np.asarray(vals)


def score_topk(models, spec, pool, k, precision="fp64", var_floor=1e-15):
    """The k best candidates of the whole pool by one unpruned scoring pass (`ombo_score_topk`): (values (k,),
    global indices (k,)) as numpy arrays, values descending, ties to the lowest index, NaN ranked as -inf.  The values
    are the ones `score(..., want_acq=True)` writes.  Slots beyond pool.m hold (-inf, -1)."""
    models, dev = _checked_models(models, pool)
    k = int(k)
    if not 1 <= k <= _cabi.TOPK_MAX:
        raise ValueError(f"k must be in 1..{_cabi.TOPK_MAX} (got {k})")
    if spec.n_models > len(models):
        raise ValueError(f"acquisition needs {spec.n_models} models, got {len(models)}")
    precision = resolve_precision(models, precision)
    G = len(models)
    gps = (_cabi.Gp * G)(*[m.c_struct(var_floor) for m in models])
    p = pool.c_struct()
    a = spec.c_struct(dev)
    out = torch.empty((k, 2), dtype=torch.int64, device=dev)
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_score_topk(ctx.handle, gps, G, C.byref(p), C.byref(a), _PREC[precision], k,
                                                C.c_void_p(out.data_ptr()), current_stream_ptr(dev)))
    host = out.cpu()
    return host[:, 0].contiguous().view(torch.float64).numpy(), host[:, 1].numpy()


def gather_rows(pool, indices, device=None):
    """Rows of the listed global indices as an explicit pool of the pool's dtype (`ombo_pool_gather`): scoring it
    reproduces the full pool's values at those indices bit for bit."""
    dev = pool.X.device if pool.X is not None else _as_device(device)
    idx = torch.as_tensor(np.asarray(indices, dtype=np.int64), device=dev)
    out = torch.empty((len(idx), pool.d), dtype=torch.float64, device=dev)
    ctx = _cabi.Context.get(dev.index)
    p = pool.c_struct()
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_pool_gather(ctx.handle, C.byref(p), C.c_void_p(idx.data_ptr()), len(idx),
                                                 C.c_void_p(out.data_ptr()), current_stream_ptr(dev)))
    if pool.X is not None and pool.X.dtype == torch.float32:
        out = out.to(torch.float32)                      # f32 values, exact in f64 and back
    return CandidatePool.explicit(out)


def top_candidates(models, spec, pool, k, precision="fp64", head=1 << 18):
    """The k best candidates among the first `head` rows of `pool` (head=None: the whole pool) as (X (k, d) ndarray,
    values (k,)), by `score_topk`.  Used to seed `polish` next to the pool winner."""
    models = _models_list(models)
    dev = models[0].device
    m = pool.m if head is None else min(pool.m, head)
    sub = CandidatePool(m=m, d=pool.d, X=None if pool.X is None else pool.X[:m], lo=pool.lo, hi=pool.hi, seed=pool.seed,
                        index_base=pool.index_base)
    vals, idx = score_topk(models, spec, sub, min(k, m), precision=precision)
    rows = torch.stack([sub.rows(int(i), 1, device=dev)[0] for i in idx])
    return rows.cpu().numpy(), vals


def propose(models, spec, pool, precision="fp64", refine_rounds=0, refine_candidates=1 << 14, refine_shrink=0.125,
            polish_top_k=0, polish_iters=30):
    """Scores the pool and returns (x_best (d,) ndarray, -acq_best, global_index), mirroring
    `(res.x, res.fun)` of the reference's `differential_evolution(obj, bounds)` call sites.

    Two refinements of the winner (SURVEY section 8f rank 3), both with the same scoring kernels:
    * refine_rounds > 0: zoom -- each round scores `refine_candidates` fresh points in a box shrunk by `refine_shrink`
      around the incumbent (clipped to the pool's box) and keeps the better point;
    * polish_top_k > 0: DE's `polish=True` (optimisers.py:118 defaults) -- bounded L-BFGS-B from the pool winner and the
      next best `polish_top_k - 1` candidates of the pool head, gradients by batched finite differences on the GPU
      (`polish`).
    The returned index is -1 once a refined point wins."""
    models = _models_list(models)
    precision = resolve_precision(models, precision)
    r = score(models, spec, pool, precision=precision)
    dev = models[0].device
    x = pool.rows(r.best_index, 1, device=dev)[0].cpu().numpy()
    best, index = r.best_value, r.best_index
    if refine_rounds > 0 and pool.lo is not None:
        lo, hi = pool.lo, pool.hi
        width = hi - lo
        for k in range(1, refine_rounds + 1):
            half = 0.5 * width * (refine_shrink ** k)
            blo, bhi = np.maximum(lo, x - half), np.minimum(hi, x + half)
            sub = CandidatePool.counter(refine_candidates, blo, bhi, seed=pool.seed + 7919 * k)
            rr = score(models, spec, sub, precision=precision)
            if rr.best_value > best:
                best, index = rr.best_value, -1
                x = sub.rows(rr.best_index, 1, device=dev)[0].cpu().numpy()
    if polish_top_k > 0 and pool.lo is not None:
        starts = x[None, :]
        if polish_top_k > 1:
            extra, _ = top_candidates(models, spec, pool, polish_top_k - 1, precision=precision)
            starts = np.vstack([starts, extra])
        xp, vp, _ = polish(models, spec, starts, pool.lo, pool.hi, max_iter=polish_iters)
        # compare in the arithmetic the polish ran in (FP64); the pool winner's own value is vals[0] >= its start value
        if vp > float(evaluate(models, spec, x[None, :], precision="fp64")[0]):
            x, best, index = xp, vp, -1
    return x, -best, index


# Kriging believer: after believing y = mu(x) at the picked x, no candidate's value rises for these kinds (the mean is
# unchanged, every variance can only fall, the front / incumbent can only improve and the value is non-decreasing in
# every sigma), so the top of the last full pass certifies later picks (DESIGN.md section 4, "Batch proposals")
_CERT_TAU = {"fast": 2e-3, "fp64": 2e-6}      # twice the acquisition contract of each precision mode
BATCH_SHORTLIST = 4096


# EHVI_BOX_FEAS is not: the probability of feasibility rises where a constraint's sigma falls with its mean above 0
def _certifiable(spec):
    return (spec.kind in (_cabi.ACQ_EI, _cabi.ACQ_EHVI_BOX)
            or (spec.kind == _cabi.ACQ_EHVI2D and spec.semantics == "exact"))


def _best_new(vals, idx):
    """(value, position) of the largest value, NaN as -inf, ties to the lowest global index."""
    v = np.where(np.isnan(vals), -np.inf, vals)
    top = v.max()
    pos = np.flatnonzero(v == top)
    return top, int(pos[np.argmin(idx[pos])])


def propose_batch(models, spec_for, pool, q, precision="fp64", shortlist=BATCH_SHORTLIST):
    """q proposals from one pool by the Kriging believer: step j believes y = mu(x_{j-1}) (the FP64 mean of the current
    models), conditions every model on it (`GPModel.with_observations`) and picks the best candidate not selected yet.

    `spec_for(Y_believed)` maps the believed objective rows so far, (j, n_models), to the AcquisitionSpec of step j;
    `spec_for(empty)` is the ordinary spec.  Step 0 is one `score_topk` pass with k = shortlist.  For EI, exact 2-D EHVI
    and box EHVI a later step first rescores only that shortlist; its best value certifies the pick when it is at
    least v_K + tau * v_1 (v_1, v_K: first and K-th values of the last full pass, tau twice the precision mode's
    acquisition contract), because no value outside the shortlist can have risen above v_K.  Otherwise, and for every
    other kind, the step runs a full pass with the fantasy models, whose top becomes the new shortlist.  The result
    is the brute-force Kriging-believer selection either way.

    Returns (X (q, d) ndarray, neg_values (q,), global indices (q,), certified (q,) bool); certified[j] is True when
    step j was decided by the shortlist alone (never for step 0).  Every point is a pool row."""
    models = _models_list(models)
    precision = resolve_precision(models, precision)
    dev = models[0].device
    q, K = int(q), int(shortlist)
    if not 1 <= q <= min(pool.m, _cabi.TOPK_MAX - 1):
        raise ValueError(f"q must be in 1..min(pool.m, {_cabi.TOPK_MAX - 1}) (got {q}, pool.m={pool.m})")
    if not 1 <= K <= _cabi.TOPK_MAX:
        raise ValueError(f"shortlist must be in 1..{_cabi.TOPK_MAX} (got {K})")
    tau = _CERT_TAU[precision]
    Y_bel = np.empty((0, len(models)))
    spec = spec_for(Y_bel)
    picked, values, certified = [], [], []

    def full_pass():
        vals, idx = score_topk(models, spec, pool, min(K + len(picked), _cabi.TOPK_MAX), precision=precision)
        keep = (idx >= 0) & ~np.isin(idx, picked)
        # every candidate outside the list ranks at or below its last entry (-inf once the list covers the pool)
        v_last = vals[-1] if idx[-1] >= 0 else -np.inf
        return vals[keep], idx[keep], vals[0], v_last

    short_v, short_i, v1, vK = full_pass()
    for j in range(q):
        if j > 0:
            x_prev = pool.rows(picked[-1], 1, device=dev)
            mu, _ = posterior(models, x_prev, precision="fp64")
            y = mu[:, 0].cpu().numpy()
            Y_bel = np.vstack([Y_bel, y[None, :]])
            models = [mdl.with_observations(x_prev, y[g:g + 1]) for g, mdl in enumerate(models)]
            spec = spec_for(Y_bel)
            ok = False
            if _certifiable(spec):
                live = ~np.isin(short_i, picked)
                if live.any():
                    cand = short_i[live]
                    new = score(models, spec, gather_rows(pool, cand, dev), precision=precision, want_acq=True,
                                want_best=False).acq.cpu().numpy()
                    best, pos = _best_new(new, cand)
                    ok = bool(best >= vK + tau * abs(v1))
            if ok:
                pick, value = int(cand[pos]), float(best)
            else:
                short_v, short_i, v1, vK = full_pass()
                pick, value = int(short_i[0]), float(short_v[0])
        else:
            ok = False
            pick, value = int(short_i[0]), float(short_v[0])
        picked.append(pick)
        values.append(value)
        certified.append(ok)
    X = np.vstack([pool.rows(i, 1, device=dev).cpu().numpy() for i in picked])
    return X, -np.asarray(values), np.asarray(picked, dtype=np.int64), np.asarray(certified)


def propose_host(models, spec, X_host, precision="fp64", index_base=0):
    """End-to-end entry: candidates live in HOST memory (numpy array or CPU tensor; pinned for
    full speed).  Chunks are copied host->device inside the call, overlapped with scoring, and
    the 16-byte result is read back.  Returns (best_value, best_global_index)."""
    models = _models_list(models)
    dev = models[0].device
    precision = resolve_precision(models, precision)
    if torch.is_tensor(X_host):
        if X_host.is_cuda:
            raise ValueError("propose_host takes host memory")
        Xh = X_host.contiguous()
        dtype = 0 if Xh.dtype == torch.float64 else 1
        if Xh.dtype not in (torch.float64, torch.float32):
            raise TypeError("host candidates must be float64 or float32")
        ptr, m, d = Xh.data_ptr(), Xh.shape[0], Xh.shape[1]
    else:
        Xh = np.ascontiguousarray(X_host)
        if Xh.dtype not in (np.float64, np.float32):
            Xh = Xh.astype(np.float64)
        dtype = 0 if Xh.dtype == np.float64 else 1
        ptr, m, d = Xh.ctypes.data, Xh.shape[0], Xh.shape[1]
    pool = CandidatePool(m=m, d=d, index_base=index_base)
    G = len(models)
    gps = (_cabi.Gp * G)(*[mm.c_struct(1e-15) for mm in models])
    p = pool.c_struct(host_ptr=ptr, host_dtype=dtype)
    a = spec.c_struct(dev)
    out = _cabi.Best()
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_score_host(ctx.handle, gps, G, C.byref(p), C.byref(a), _PREC[precision],
                                                C.byref(out), current_stream_ptr(dev)))
    return float(out.value), int(out.index)


# --------------------------------------------------------------------------------------------
# batched twins of the reference's acquisition callables (same names and argument order)
# --------------------------------------------------------------------------------------------
def EHVI(X, models, max_point, PF, cache, semantics="reference", precision="fp64"):
    return evaluate(models, spec_ehvi(max_point, PF, cache, semantics), X, precision)


def EHVI_3D(X, models, max_point, PF, cache, semantics="reference", precision="fp64"):
    return evaluate(models, spec_ehvi3d(max_point, PF, cache, semantics), X, precision)


def EHVI_box(X, models, max_point, PF, precision="fp64"):
    return evaluate(models, spec_ehvi_box(max_point, PF), X, precision)


def EHVI_box_feasible(X, models, constraint_models, max_point, PF, precision="fp64"):
    models = list(_models_list(models)) + list(constraint_models)
    k = len(np.asarray(max_point).reshape(-1))
    return evaluate(models, spec_ehvi_box_feasible(max_point, PF, len(models) - k), X, precision)


def expected_decomposition(X, models, weights, agg_func, agg_function_min, cache, semantics="reference",
                           precision="fp64"):
    return evaluate(models, spec_expected_decomposition(weights, agg_func, agg_function_min, cache, semantics),
                    X, precision)


def expected_improvement(X, model, opt_value, var_eps=0.0, precision="fp64"):
    return evaluate([model], spec_ei(opt_value, var_eps), X, precision)


def consraint_ei(X, aggregate_model, constraint_models, current_best, precision="fp64"):
    models = [aggregate_model] + list(constraint_models)
    return evaluate(models, spec_constrained_ei(current_best, len(constraint_models)), X, precision)


def pareto_expected_improvement(X, pareto_model, scalarised_model, opt_value, precision="fp64"):
    return evaluate([pareto_model, scalarised_model], spec_pareto_ei(opt_value), X, precision)


def hypervolume_based_PoI(X, models, P, cells, precision="fp64"):
    return evaluate(models, spec_hv_poi(cells), X, precision)


def hypervolume_based_PoI_box(X, models, ideal_point, max_point, PF, precision="fp64"):
    return evaluate(models, spec_hv_poi_box(ideal_point, max_point, PF), X, precision)
