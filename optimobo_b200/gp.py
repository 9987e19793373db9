"""GP surrogate whose posterior is evaluated by the CUDA hot path.

`GPModel` stands where the reference puts a `GPy.models.GPRegression(X, y, Matern52(ARD))`
(optimobo/algorithms/optimisers.py:226-231 and the other sites listed in SURVEY.md section 0.1)
and answers BOTH model surfaces the reference calls (SURVEY section 8b):

  * GPy:     predict(Xnew (m,d))            -> (mean (m,1), var (m,1))   variance clipped at 1e-15
  * sklearn: predict(X, return_std=True)    -> (mean (m,),  std (m,))    negative variance -> 0
             (util_functions.py:265)

so the reference's own `util_functions.EHVI` etc. run unmodified on it.  PyTorch tensors hold
the training set and the state blob (L, L^-1, alpha, fast-path planes); all arithmetic happens
in liboptimobo_b200.so.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import types

import numpy as np
import torch

from . import _cabi

_KERNELS = {"matern52": _cabi.KERNEL_MATERN52, "rbf": _cabi.KERNEL_RBF}


def _as_device(device):
    dev = torch.device(device if device is not None else "cuda:0")
    if dev.type != "cuda":
        raise RuntimeError("optimobo_b200 runs on CUDA devices only (no CPU fallback)")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def current_stream_ptr(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


class GPModel:
    """Exact GP regression state (zero-mean, no y-normalisation, like GPRegression's defaults)."""

    def __init__(self, X, y, lengthscale, variance=1.0, noise=0.0, jitter=1e-8, kernel="matern52",
                 device=None, refresh=True, max_jitter_tries=6):
        self.device = _as_device(device)
        self.X = torch.as_tensor(np.asarray(X, dtype=np.float64) if not torch.is_tensor(X) else X,
                                 dtype=torch.float64).to(self.device).contiguous()
        if self.X.dim() != 2:
            raise ValueError("X must be (n, d)")
        self.y = torch.as_tensor(np.asarray(y, dtype=np.float64) if not torch.is_tensor(y) else y,
                                 dtype=torch.float64).to(self.device).reshape(-1).contiguous()
        self.n, self.d = self.X.shape
        if self.y.numel() != self.n:
            raise ValueError("y must have one value per row of X")
        if kernel not in _KERNELS:
            raise ValueError(f"unknown kernel {kernel!r} (matern52 | rbf)")
        self.kernel_name = kernel
        self.kernel = _KERNELS[kernel]
        self.lengthscale = np.broadcast_to(np.asarray(lengthscale, dtype=np.float64), (self.d,)).copy()
        self.variance = float(variance)
        self.noise = float(noise)
        self.jitter = float(jitter)
        self.max_jitter_tries = max_jitter_tries
        self.n_pad = _cabi.lib().ombo_n_pad(self.n)
        self.state = torch.empty(_cabi.state_bytes(self.n, self.d), dtype=torch.uint8, device=self.device)
        # read by TuRBO in the reference (turbo.py:83); kept for surface compatibility
        self.kern = types.SimpleNamespace(lengthscale=self.lengthscale, variance=self.variance)
        self.refreshed = False
        self._conditioning = None
        if refresh:
            self.refresh()

    # ---- K3 ------------------------------------------------------------------------------
    def refresh(self):
        """(Re)builds L, L^-1, alpha on the device.  On a non-PD matrix the jitter is raised
        x10 per try starting from mean(diag K) * 1e-6, like GPy's jitchol."""
        ctx = _cabi.Context.get(self.device.index)
        ell = (C.c_double * self.d)(*self.lengthscale.tolist())
        jitter = self.jitter
        for attempt in range(self.max_jitter_tries + 1):
            spec = _cabi.GpSpec(n=self.n, d=self.d, kernel=self.kernel, reserved=2 | 4,   # fp16 and f8c planes allowed
                                sigma_f2=self.variance, sigma_n2=self.noise, jitter=jitter,
                                X=self.X.data_ptr(), y=self.y.data_ptr(), ell=ell)
            with torch.cuda.device(self.device):
                rc = _cabi.lib().ombo_gp_refresh(ctx.handle, C.byref(spec), C.c_void_p(self.state.data_ptr()),
                                                 current_stream_ptr(self.device))
            if rc == _cabi.ERR_NOT_PD and attempt < self.max_jitter_tries:
                base = (self.variance + self.noise) * 1e-6
                jitter = base if jitter < base else jitter * 10.0
                continue
            _cabi.check(rc)
            break
        self.effective_jitter = jitter
        self.refreshed = True
        self._conditioning = None
        # word 1 of the status field: format of the fast mode's operand planes the refresh stored
        # (0 bf16 x3, 1 fp16 x3, 2 "f8c" = fp16 + two e4m3 correction planes) -> ombo_gp.reserved flags
        st = self._field(_cabi.FIELD_STATUS, torch.int32, (4,)).cpu()
        self.plane_format = ("bf16x3", "fp16x3", "f8c")[int(st[1])]
        self._flags = (0, 2, 4)[int(st[1])]           # OMBO_GP_FP16_PLANES / OMBO_GP_F8C_PLANES
        return self

    def with_observations(self, X_new, y_new):
        """A new model with the rows (X_new, y_new) appended: the same hyper-parameters, kernel, noise and jitter
        policy, refreshed by K3.  This model's X / y are not mutated (Kriging-believer batches condition on
        y_new = mu(X_new))."""
        Xn = torch.as_tensor(X_new, dtype=torch.float64).to(self.device).reshape(-1, self.d)
        yn = torch.as_tensor(y_new, dtype=torch.float64).to(self.device).reshape(-1)
        return GPModel(torch.cat([self.X, Xn]), torch.cat([self.y, yn]), self.lengthscale, self.variance,
                       noise=self.noise, jitter=self.jitter, kernel=self.kernel_name, device=self.device,
                       max_jitter_tries=self.max_jitter_tries)

    # fast precision mode keeps sigma within 1e-3 sigma_f while `conditioning` stays below this (measured,
    # scripts/cond_study.py: the error grows from 4e-5 sigma_f at 15 to 2.4e-4 at 4e2, 1e-3 at 4e3-8e3, 1.5e-2 at 4e7)
    FAST_MODE_CONDITIONING_LIMIT = 2.0e3

    @property
    def conditioning(self):
        """(max L_ii / min L_ii)^2 of the Cholesky factor: a cheap proxy of cond(K) (one 8-byte readback,
        cached until the next refresh).  The split-precision fast mode loses absolute accuracy on sigma
        roughly in proportion to its square root, because V = L^-1 k* is then a sum of large cancelling
        terms."""
        if self._conditioning is None:
            dg = torch.diagonal(self._field(_cabi.FIELD_L, torch.float64, (self.n_pad, self.n_pad)))[: self.n]
            self._conditioning = float((dg.max() / dg.min()) ** 2)
        return self._conditioning

    def _field(self, field, dtype, shape):
        off, cnt = _cabi.state_field(self.n, self.d, field)
        esz = torch.empty((), dtype=dtype).element_size()
        return self.state[off:off + cnt * esz].view(dtype).view(*shape)

    @property
    def L(self):
        # only the lower triangle of the working matrix is the factor (the strict upper blocks
        # still hold K)
        return torch.tril(self._field(_cabi.FIELD_L, torch.float64, (self.n_pad, self.n_pad))[: self.n, : self.n])

    @property
    def Linv(self):
        return self._field(_cabi.FIELD_LINV, torch.float64, (self.n_pad, self.n_pad))[: self.n, : self.n]

    @property
    def alpha(self):
        return self._field(_cabi.FIELD_ALPHA, torch.float64, (self.n_pad,))[: self.n]

    def c_struct(self, var_floor=1e-15):
        if not self.refreshed:
            raise RuntimeError("GPModel.refresh() has not been run")
        # reserved = flags of the refreshed state (format of the fast mode's operand planes)
        return _cabi.Gp(n=self.n, d=self.d, kernel=self.kernel, reserved=self._flags, sigma_f2=self.variance,
                        sigma_n2=self.noise, var_floor=var_floor, state=self.state.data_ptr())

    # ---- the two model surfaces ------------------------------------------------------------
    def predict(self, Xnew, return_std=False, precision="fp64"):
        from .acquisition import posterior
        Xn = np.atleast_2d(np.asarray(Xnew.detach().cpu() if torch.is_tensor(Xnew) else Xnew, dtype=np.float64))
        mu, var = posterior([self], Xn, precision=precision, var_floor=0.0 if return_std else 1e-15)
        mu = mu[0].cpu().numpy()
        var = var[0].cpu().numpy()
        if return_std:
            return mu, np.sqrt(np.maximum(var, 0.0))
        return mu.reshape(-1, 1), var.reshape(-1, 1)

    def posterior_samples(self, X, size=10, rng=None, jitter=None, max_jitter_tries=6):
        """Joint posterior samples at X (m,d) -> (m, 1, size), GPy's `posterior_samples` shape
        (turbo.py:116).  out = mu + chol(Sigma + (noise + jitter) I) Z with Z ~ N(0, I) drawn from `rng`
        on the host; covariance, Cholesky and the product run on the device in FP64
        (`ombo_posterior_joint_samples`).  The jitter starts at 1e-8 sigma_f^2 and is raised x10 while the
        posterior covariance is not numerically positive definite (GPy's jitchol policy)."""
        Z = (np.random.default_rng() if rng is None else rng).standard_normal((len(np.atleast_2d(X)), int(size)))
        return self.posterior_samples_from(X, Z, jitter, max_jitter_tries)

    posterior_samples_f = posterior_samples      # noise is fixed to 0 on this path (optimisers.py:229)

    def posterior_samples_from(self, X, Z, jitter=None, max_jitter_tries=6):
        """As `posterior_samples`, with the standard-normal draws Z (m, size) supplied (parity tests)."""
        Xd = torch.as_tensor(np.ascontiguousarray(np.atleast_2d(np.asarray(X, dtype=np.float64)))).to(self.device)
        Zd = torch.as_tensor(np.ascontiguousarray(np.asarray(Z, dtype=np.float64))).to(self.device)
        m, S = Zd.shape
        if Xd.shape != (m, self.d):
            raise ValueError(f"X must be ({m}, {self.d}), got {tuple(Xd.shape)}")
        out = torch.empty((m, S), dtype=torch.float64, device=self.device)
        ctx = _cabi.Context.get(self.device.index)
        g = self.c_struct()
        jit = 1e-8 * self.variance if jitter is None else float(jitter)
        for attempt in range(max_jitter_tries + 1):
            with torch.cuda.device(self.device):
                rc = _cabi.lib().ombo_posterior_joint_samples(
                    ctx.handle, C.byref(g), C.c_void_p(Xd.data_ptr()), m, C.c_void_p(Zd.data_ptr()), S,
                    self.noise + jit, C.c_void_p(out.data_ptr()), current_stream_ptr(self.device))
            if rc == _cabi.ERR_NOT_PD and attempt < max_jitter_tries:
                jit = max(jit, 1e-10 * self.variance) * 10.0
                continue
            _cabi.check(rc)
            break
        self.sample_jitter = jit
        return out.cpu().numpy().reshape(m, 1, S)

    @classmethod
    def from_gpy(cls, gpy_model, device=None):
        """Adopts the hyper-parameters of a fitted GPy GPRegression (reference models)."""
        kern = gpy_model.kern
        return cls(np.asarray(gpy_model.X), np.asarray(gpy_model.Y).reshape(-1),
                   np.asarray(kern.lengthscale), float(np.asarray(kern.variance).reshape(-1)[0]),
                   noise=float(np.asarray(gpy_model.Gaussian_noise.variance).reshape(-1)[0]), device=device)


_REFRESH_STREAMS = {}
_REFRESH_POOL = None          # host threads are kept: starting two per call costs as much as the overlap saves


def refresh_models(models):
    """Refreshes several GPs of one device concurrently.  K3 is a chain of small dependent launches (16 diagonal
    blocks of one CTA each at n = 1024) that leaves most SMs idle, so the models' chains overlap on separate streams:
    2 GPs at n = 1024 take about the time of one.  One host thread per model, because the C entry synchronises its
    stream to read the positive-definiteness flag (ctypes drops the GIL for the call).  State blobs are per model, the
    context holds no refresh workspace, so the calls share nothing but the launch counter."""
    models = list(models)
    if len(models) <= 1 or len({m.device for m in models}) != 1:
        for m in models:
            m.refresh()
        return models
    global _REFRESH_POOL
    if _REFRESH_POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _REFRESH_POOL = ThreadPoolExecutor(max_workers=8, thread_name_prefix="ombo-refresh")
    dev = models[0].device
    pool = _REFRESH_STREAMS.setdefault(dev, [])
    while len(pool) < len(models):
        pool.append(torch.cuda.Stream(dev))
    cur = torch.cuda.current_stream(dev)
    for st in pool[: len(models)]:
        st.wait_stream(cur)

    def work(arg):
        m, st = arg
        with torch.cuda.device(dev), torch.cuda.stream(st):
            m.refresh()

    list(_REFRESH_POOL.map(work, zip(models, pool)))
    for st in pool[: len(models)]:
        cur.wait_stream(st)
    return models
