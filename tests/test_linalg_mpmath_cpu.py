"""The mpmath reference of the FP64 factorisations (tests/linalg_mpmath.py) checked on its own, without a GPU: rounded
to float64 it agrees with LAPACK and with the float64 oracle where the problem is well conditioned, its analytic
likelihood gradient agrees with central differences of its own likelihood (with and without noise), and with the host
fit's float64 derivation where the noise is zero."""
import mpmath as mp
import numpy as np
import pytest
from scipy import linalg as sla

import linalg_mpmath as R
from oracle import oracle as O
from optimobo_b200.fit import _nlml_and_grad

U = 2.0 ** -53


def _problem(n, d, seed, spread=1.0):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d)) * spread
    y = np.sin(3 * X[:, 0]) + X[:, -1] ** 2 + 0.1 * rng.standard_normal(n)
    ell = rng.uniform(0.3, 0.9, d)
    return X, y, ell


def _okern(kernel):
    return O.KERNEL_MATERN52 if kernel == R.MATERN52 else O.KERNEL_RBF


@pytest.mark.parametrize("n,d,kernel,sn2", [(1, 1, R.MATERN52, 0.0), (17, 3, R.MATERN52, 0.0), (40, 5, R.RBF, 1e-2),
                                            (65, 2, R.MATERN52, 1e-2)])
def test_reference_factor_matches_lapack(n, d, kernel, sn2):
    """L, L^-1 and alpha rounded to float64 against scipy's cholesky / solve_triangular / cho_solve of the same K:
    both are within c n u kappa of the exact factor, and these shapes have kappa <= ~1e4."""
    X, y, ell = _problem(n, d, n)
    xs = X / ell
    K, L, Linv, a = R.factor(xs, y, 1.3, kernel, sn2, 1e-8)
    Kf = R.to_np(K)
    kappa = R.cond2(K)
    assert kappa < 1e6
    Kd = O.k_of_r(O.scaled_dist(X, X, ell, "direct"), 1.3, _okern(kernel)) + (sn2 + 1e-8) * np.eye(n)
    # the same matrix: the float64 oracle rounds ~10 times per entry (sum, sqrt, polynomial, exp, products)
    np.testing.assert_allclose(Kf, Kd, rtol=16 * U, atol=0)
    Ls = sla.cholesky(Kf, lower=True)
    tol = 8 * n * U * kappa
    assert np.linalg.norm(R.to_np(L) - Ls) <= tol * np.linalg.norm(Ls)
    Xs = sla.solve_triangular(Ls, np.eye(n), lower=True)
    assert np.linalg.norm(R.to_np(Linv) - Xs) <= tol * np.sqrt(kappa) * np.linalg.norm(Xs)
    As = sla.cho_solve((Ls, True), y)
    assert np.linalg.norm(R.to_np(a) - As) <= tol * np.linalg.norm(As)
    # the reference itself: L L^T = K and L^-1 L = I to its own 40 digits
    Lm, Xm = mp.matrix(L), mp.matrix(Linv)
    assert mp.mnorm(Lm * Lm.T - mp.matrix(K), 1) <= mp.mpf(10) ** -30 * mp.mnorm(mp.matrix(K), 1)
    assert mp.mnorm(Xm * Lm - mp.eye(n), 1) <= mp.mpf(10) ** -30 * kappa


@pytest.mark.parametrize("n,d,m,kernel,sn2", [(10, 2, 7, R.MATERN52, 0.0), (30, 3, 20, R.RBF, 1e-2)])
def test_reference_joint_sigma_matches_oracle(n, d, m, kernel, sn2):
    X, y, ell = _problem(n, d, 3)
    Xc = np.random.default_rng(4).random((m, d))
    st = O.gp_fit_state(X, y, ell, 0.8, sigma_n2=sn2, jitter=1e-8, kernel=_okern(kernel), form="direct")
    mu_o, S_o = O.gp_posterior_joint(st, Xc)
    S = R.to_np(R.joint_sigma(X / ell, Xc / ell, 0.8, kernel, sn2 + 1e-8))
    K = R.kernel_matrix(X / ell, 0.8, kernel, sn2, 1e-8)
    bound = 16 * n * U * R.cond2(K) * 0.8                     # |Sigma error| <= c n u kappa(K) |K**| (K** <= sigma_f2)
    np.testing.assert_allclose(S, S_o, rtol=0, atol=bound)
    mu = R.to_np(R.joint_mean(X / ell, y, Xc / ell, 0.8, kernel, sn2 + 1e-8))
    # mu = K*^T alpha: the error of alpha (c n u kappa |alpha|) through a row of K* (entries <= sigma_f2)
    np.testing.assert_allclose(mu, mu_o, rtol=0, atol=16 * n * U * R.cond2(K) * 0.8 * np.abs(st["alpha"]).sum())


@pytest.mark.parametrize("n,d,kernel,sn2", [(6, 2, R.MATERN52, 0.0), (6, 2, R.MATERN52, 0.05), (9, 3, R.RBF, 0.0),
                                            (9, 3, R.RBF, 0.05), (1, 2, R.MATERN52, 0.05)])
def test_reference_gradient_matches_central_differences(n, d, kernel, sn2):
    """Central differences of the reference's own NLML, all in mpmath: h = 1e-12 leaves a truncation error of
    ~h^2 |f'''| ~ 1e-24, far below the 1e-15 the comparison asks for."""
    X, y, ell = _problem(n, d, 7)
    xs, sf2 = X / ell, 1.7
    f, g = R.nlml_grad(xs, y, sf2, kernel, sn2, 1e-8)
    assert abs(f - R.nlml(xs, y, sf2, kernel, sn2, 1e-8)) <= mp.mpf(10) ** -30 * (1 + abs(f))
    h = mp.mpf(10) ** -12
    one = [mp.mpf(1)] * d
    fd = [(R.nlml(xs, y, sf2 * mp.exp(h), kernel, sn2, 1e-8) - R.nlml(xs, y, sf2 * mp.exp(-h), kernel, sn2, 1e-8)) / (2 * h)]
    for t in range(d):
        up, dn = list(one), list(one)
        up[t], dn[t] = mp.exp(-h), mp.exp(h)                  # log ell_t +- h scales column t of xs by exp(-+h)
        fd.append((R.nlml(xs, y, mp.mpf(sf2), kernel, sn2, 1e-8, up) - R.nlml(xs, y, mp.mpf(sf2), kernel, sn2, 1e-8, dn))
                  / (2 * h))
    scale = max(abs(v) for v in g) + 1
    for a, b in zip(g, fd):
        assert abs(a - b) <= mp.mpf(10) ** -15 * scale, (a, b)


@pytest.mark.parametrize("n,d,kernel", [(12, 2, R.MATERN52), (25, 4, R.RBF), (40, 3, R.MATERN52)])
def test_reference_nlml_matches_host_fit(n, d, kernel):
    """The host fit's float64 derivation (sigma_n2 = 0, jitter 1e-8) against the reference: an independent derivation
    of the same formula, equal to within c n u kappa of the value."""
    X, y, ell = _problem(n, d, 11)
    sf2 = 0.9
    theta = np.log(np.concatenate(([sf2], ell)))
    f_h, g_h = _nlml_and_grad(theta, X, y, kernel, 1e-8)
    # the host divides by exp(log ell), not by ell: use its scaled inputs so both see the same float64 matrix
    xs = X / np.exp(theta[1:])
    f, g = R.nlml_grad(xs, y, float(np.exp(theta[0])), kernel, 0.0, 1e-8)
    kappa = R.cond2(R.kernel_matrix(xs, float(np.exp(theta[0])), kernel, 0.0, 1e-8))
    tol = 16 * n * U * kappa
    g = R.to_np(g)
    assert abs(f_h - float(f)) <= tol * (abs(float(f)) + np.abs(y).max() ** 2 * n)
    np.testing.assert_allclose(g_h, g, rtol=0, atol=tol * (np.abs(g).max() + n * np.abs(y).max() ** 2))
