"""High-precision reference (mpmath, 50 digits) of the acquisition formulas that oracle/oracle.py restates in float64.
Only the tests import it, and it imports nothing from optimobo_b200.  Inputs are float64 arrays and are taken as exact;
every operation after that runs in mpmath, so the result is the formula's exact value rounded once to float64.  Each
call loops over the candidates in plain Python: keep the candidate counts small (about 2e5 evaluations per test run).

The formulas are the reference's, constants included (the 1e-10 in EI's denominator, the 1e-5 added to the
constraint and HV-PoI variances, the P stripes of the reference-semantics 2-D EHVI), so that the float64 oracle agrees
with this module wherever its own arithmetic is well conditioned."""
from __future__ import annotations

import mpmath as mp
import numpy as np

mp.mp.dps = 50

_F = mp.mpf


def _vec(fn, *cols):
    cols = [np.asarray(c, dtype=np.float64).reshape(-1) for c in np.broadcast_arrays(*cols)]
    out = np.empty(len(cols[0]))
    for j in range(len(out)):
        args = [c[j] for c in cols]
        out[j] = np.nan if any(np.isnan(a) for a in args) else float(fn(*[_F(a) for a in args]))
    return out


def Phi(t):
    return mp.ncdf(t)


def phi(t):
    return mp.npdf(t)


def h(t):
    """phi(t) + t Phi(t) = E[(t - z)^+] for z ~ N(0, 1): EI / sigma and psi / sigma."""
    return phi(t) + t * Phi(t)


# ---- EI family (optimisers.py:325-344, cparego.py:450-496, keep.py:142-150) ---------------------
def _ei(mu, var, best, eps):
    s = mp.sqrt(var + eps)
    g = (best - mu) / (s + _F(1e-10))
    return s * h(g)


def expected_improvement(mu, var, best, var_eps=0.0):
    return _vec(_ei, mu, var, best, var_eps)


def _pof(mu, var):
    return Phi((0 - mu) / mp.sqrt(var + _F(1e-5)))


def probability_of_feasibility(mu, var):
    return _vec(_pof, mu, var)


def constrained_ei(mu, var, best):
    """mu / var (m, 1 + n_constr), column 0 the aggregate model."""
    mu = np.atleast_2d(np.asarray(mu, float))
    var = np.atleast_2d(np.asarray(var, float))

    def one(j):
        if np.isnan(mu[j]).any() or np.isnan(var[j]).any():
            return np.nan
        v = _ei(_F(mu[j, 0]), _F(var[j, 0]), _F(best), _F(0))
        for c in range(1, mu.shape[1]):
            v *= _pof(_F(mu[j, c]), _F(var[j, c]))
        return float(v)
    return np.array([one(j) for j in range(len(mu))])


def pareto_ei(mu_pareto, mu_scalar, var_scalar, best):
    return _vec(lambda p, m, v, b: p * _ei(m, v, b, _F(1e-6)), mu_pareto, mu_scalar, var_scalar, best)


# ---- HV-PoI (emo.py:176-228) ---------------------------------------------------------------------
def hv_poi(mu, var, cells):
    """mu / var (m, >= 2); cells (n_cells, 2, 2), [c][0] upper, [c][1] lower (as spec_hv_poi takes them)."""
    mu = np.atleast_2d(np.asarray(mu, float))[:, :2]
    var = np.atleast_2d(np.asarray(var, float))[:, :2]
    cells = np.asarray(cells, float)

    def one(j):
        if np.isnan(mu[j]).any() or np.isnan(var[j]).any():
            return np.nan
        m = [_F(x) for x in mu[j]]
        s = [mp.sqrt(_F(x) + _F(1e-5)) for x in var[j]]
        poi, imp = _F(0), _F(0)
        for U, L in cells:
            p, vol, valid = _F(1), _F(1), True
            for i in range(2):
                a, b = (_F(U[i]) - m[i]) / s[i], (_F(L[i]) - m[i]) / s[i]
                # Phi(a) - Phi(b) from the small side: 50 digits cannot hold 1 - Phi(b) once b > ~15
                p *= Phi(-b) - Phi(-a) if b > 0 else Phi(a) - Phi(b)
                valid = valid and U[i] > mu[j, i]
                vol *= _F(U[i]) - max(_F(L[i]), m[i])
            poi += p
            if valid:
                imp += vol
        return float(poi * imp)
    return np.array([one(j) for j in range(len(mu))])


# ---- 2-D EHVI (util_functions.py:81-167) ---------------------------------------------------------
def _psi(a, b, m, s):
    t = (b - m) / s
    return s * phi(t) + (a - m) * Phi(t)


def ehvi2d(stripes, mu0, mu1, s0, s1, exact):
    """stripes (2, P + 2): y1, y2 as host_prep.ehvi_stripes / oracle.ehvi_stripes build them.  s0, s1 are the 'sigma'
    the formula takes: var0 * C00 and var0 * C01 in the reference semantics (P stripes), the true standard deviations
    in the exact semantics (P + 1 stripes)."""
    y1 = [_F(x) for x in stripes[0]]
    y2 = [_F(x) for x in stripes[1]]
    P = len(y1) - 2

    def one(m0, m1, a, b):
        sum1, sum2 = _F(0), _F(0)
        for i in range(1, P + 1):
            t = (y1[i] - m0) / a
            psi2 = _psi(y2[i], y2[i], m1, b)
            sum1 += (y1[i - 1] - y1[i]) * Phi(t) * psi2
            sum2 += (_psi(y1[i - 1], y1[i - 1], m0, a) - _psi(y1[i - 1], y1[i], m0, a)) * psi2
        if exact:
            sum2 += _psi(y1[P], y1[P], m0, a) * _psi(y2[P + 1], y2[P + 1], m1, b)
        return sum1 + sum2
    return _vec(one, mu0, mu1, s0, s1)


def ehvi2d_posterior(stripes, mu, var, semantics, cache_c=(0.0, 0.0)):
    """The 2-D EHVI of posteriors mu / var (m, 2) in either semantics (cache_c = (C00, C01) for the reference one)."""
    mu = np.asarray(mu, float)
    var = np.asarray(var, float)
    if semantics == "reference":
        return ehvi2d(stripes, mu[:, 0], mu[:, 1], var[:, 0] * cache_c[0], var[:, 0] * cache_c[1], False)
    return ehvi2d(stripes, mu[:, 0], mu[:, 1], np.sqrt(var[:, 0]), np.sqrt(var[:, 1]), True)


# ---- crude 3-D EHVI (util_functions.py:170-214) --------------------------------------------------
def ehvi3d(mu, var, r, sminus, cache, semantics="reference"):
    """mean_j max(0, prod_i (r_i - Y_ji) - Sminus) over the samples Y_j = cache_j * sd + mu inside the box of r."""
    mu = np.atleast_2d(np.asarray(mu, float))
    var = np.atleast_2d(np.asarray(var, float))
    cache = np.asarray(cache, float)
    k = cache.shape[1]
    rr = [_F(x) for x in r]

    def one(j):
        if np.isnan(mu[j, :k]).any() or np.isnan(var[j, :k]).any():
            return np.nan
        sd = [mp.sqrt(_F(var[j, 0] if semantics == "reference" else var[j, i])) for i in range(k)]
        total = _F(0)
        for z in cache:
            diff = [rr[i] - (_F(z[i]) * sd[i] + _F(mu[j, i])) for i in range(k)]
            if all(d >= 0 for d in diff):
                v = mp.fprod(diff) - _F(sminus)
                if v > 0:
                    total += v
        return float(total / len(cache))
    return np.array([one(j) for j in range(len(mu))])


# ---- box EHVI (not in the reference; tests/ehvi_oracle.py sums the same integrand on the full grid) --------
def expected_shortfall(t, mu, sd):
    """H(t) = E[(t - y)^+] for y ~ N(mu, sd^2); H(-inf) = 0."""
    if mp.isinf(t):
        return _F(0)
    return sd * h((t - mu) / sd)


def ehvi_box(table, boxes, mu, var):
    """table (k, B) breakpoints, boxes (n, 2, k) breakpoint indices [u, l] (host_prep.ehvi_boxes):
    sum over the boxes of prod_i (H_i(table[i, u_i]) - H_i(table[i, l_i]))."""
    table = np.asarray(table, float)
    boxes = np.asarray(boxes).astype(np.int64)
    mu = np.atleast_2d(np.asarray(mu, float))
    var = np.atleast_2d(np.asarray(var, float))
    k, B = table.shape

    def one(j):
        if np.isnan(mu[j, :k]).any() or np.isnan(var[j, :k]).any():
            return np.nan
        Hs = [[expected_shortfall(_F(table[i, b]), _F(mu[j, i]), mp.sqrt(_F(var[j, i]))) for b in range(B)]
              for i in range(k)]
        total = _F(0)
        for U, L in boxes:
            total += mp.fprod(Hs[i][U[i]] - Hs[i][L[i]] for i in range(k))
        return float(total)
    return np.array([one(j) for j in range(len(mu))])


def argmax_lowest_index(v):
    """np.argmax semantics with NaN taken as -inf."""
    v = np.where(np.isnan(v), -np.inf, np.asarray(v, float))
    return int(np.argmax(v))
