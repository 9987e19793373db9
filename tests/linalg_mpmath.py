"""High-precision reference (mpmath, 40 digits) of the FP64 factorisations under the GP: the covariance matrix K, its
Cholesky factor, L^-1, alpha = K^-1 y, the negative log marginal likelihood and its gradient, and the joint posterior
covariance of a candidate set.  Only the tests import it, and it imports nothing from optimobo_b200.

Inputs are float64 arrays and are taken as exact.  The scaled inputs xs = X / ell are formed in float64 by the caller,
because that is what the device works from (k_prepare, k_joint_scale); distances are direct differences of them, as in
k_build_K.  Every operation after that runs in mpmath, so each result is the exact value of the float64 inputs, rounded
once when converted back.  Matrices are lists of rows of mpf.  The cost is cubic in plain Python: keep n, m <= ~129
(n = 129 takes about a second per factorisation)."""
from __future__ import annotations

import mpmath as mp
import numpy as np

mp.mp.dps = 40

_F = mp.mpf
MATERN52, RBF = "matern52", "rbf"
_S5 = mp.sqrt(5)


def _mp_rows(A):
    A = np.atleast_2d(np.asarray(A, dtype=np.float64))
    return [[_F(float(v)) for v in row] for row in A]


def to_np(M):
    """Rounds an mpmath vector or matrix (list of rows) to float64 once."""
    if len(M) and isinstance(M[0], list):
        return np.array([[float(v) for v in row] for row in M], dtype=np.float64)
    return np.array([float(v) for v in M], dtype=np.float64)


def _k0_dk(r2, kernel):
    """k0(r) (the kernel at sigma_f2 = 1) and dk such that d k0 / d log ell_t = dk * (xs_it - xs_jt)^2."""
    if kernel == MATERN52:
        r = mp.sqrt(r2)
        e = mp.exp(-_S5 * r)
        return (1 + _S5 * r + _F(5) / 3 * r2) * e, _F(5) / 3 * (1 + _S5 * r) * e
    k0 = mp.exp(-r2 / 2)
    return k0, k0


def _diff2(a, b):
    return [(u - v) ** 2 for u, v in zip(a, b)]


def cross_kernel(xa, xb, sf2, kernel):
    """k(a_i, b_j) for the scaled inputs xa (na, d), xb (nb, d)."""
    A, B, s = _mp_rows(xa), _mp_rows(xb), _F(sf2)
    return [[s * _k0_dk(mp.fsum(_diff2(a, b)), kernel)[0] for b in B] for a in A]


def kernel_matrix(xs, sf2, kernel, sn2=0.0, jitter=0.0):
    """K = k(xs, xs) + (sigma_n2 + jitter) I, the matrix k_build_K forms (symmetric: each pair evaluated once)."""
    P, s = _mp_rows(xs), _F(sf2)
    n = len(P)
    K = [[None] * n for _ in range(n)]
    for i in range(n):
        for j in range(i + 1):
            K[i][j] = K[j][i] = s * _k0_dk(mp.fsum(_diff2(P[i], P[j])), kernel)[0]
        K[i][i] += _F(sn2) + _F(jitter)
    return K


def cholesky(K):
    """Lower-triangular L with L L^T = K (zeros above the diagonal); raises ValueError if K is not positive definite."""
    n = len(K)
    L = [[_F(0)] * n for _ in range(n)]
    for j in range(n):
        p = K[j][j] - mp.fdot(L[j][:j], L[j][:j])
        if p <= 0:
            raise ValueError(f"not positive definite at row {j}")
        L[j][j] = mp.sqrt(p)
        for i in range(j + 1, n):
            L[i][j] = (K[i][j] - mp.fdot(L[i][:j], L[j][:j])) / L[j][j]
    return L


def tri_inv(L):
    """X = L^-1 by forward substitution, column by column (L X = I); about the cost of the Cholesky."""
    n = len(L)
    X = [[_F(0)] * n for _ in range(n)]
    for c in range(n):
        X[c][c] = 1 / L[c][c]
        for i in range(c + 1, n):
            X[i][c] = -mp.fdot(L[i][c:i], [X[k][c] for k in range(c, i)]) / L[i][i]
    return X


def forward(L, b):
    """L^-1 b for a vector b."""
    x = []
    for i in range(len(L)):
        x.append((b[i] - mp.fdot(L[i][:i], x)) / L[i][i])
    return x


def backward_t(L, b):
    """L^-T b for a vector b."""
    n = len(L)
    x = [_F(0)] * n
    for i in range(n - 1, -1, -1):
        x[i] = (b[i] - mp.fdot([L[k][i] for k in range(i + 1, n)], x[i + 1:])) / L[i][i]
    return x


def alpha(L, y):
    """alpha = K^-1 y = L^-T L^-1 y."""
    return backward_t(L, forward(L, [_F(float(v)) for v in np.asarray(y, np.float64)]))


def factor(xs, y, sf2, kernel, sn2=0.0, jitter=0.0):
    """(K, L, L^-1, alpha) of one GP."""
    K = kernel_matrix(xs, sf2, kernel, sn2, jitter)
    L = cholesky(K)
    return K, L, tri_inv(L), alpha(L, y)


def nlml(xs, y, sf2, kernel, sn2=0.0, jitter=0.0, xs_scale=None):
    """1/2 y^T K^-1 y + sum log L_ii + n/2 log(2 pi).  xs_scale (d,) optional mpf factors applied to the columns of xs
    after the conversion (central differences in log ell at fixed float64 inputs); sf2 may be an mpf."""
    P = _mp_rows(xs)
    if xs_scale is not None:
        P = [[v * s for v, s in zip(row, xs_scale)] for row in P]
    s = sf2 if isinstance(sf2, mp.mpf) else _F(sf2)
    n = len(P)
    K = [[None] * n for _ in range(n)]
    for i in range(n):
        for j in range(i + 1):
            K[i][j] = K[j][i] = s * _k0_dk(mp.fsum(_diff2(P[i], P[j])), kernel)[0]
        K[i][i] += _F(sn2) + _F(jitter)
    L = cholesky(K)
    yv = [_F(float(v)) for v in np.asarray(y, np.float64)]
    t = forward(L, yv)
    return mp.fdot(t, t) / 2 + mp.fsum(mp.log(L[i][i]) for i in range(n)) + n * mp.log(2 * mp.pi) / 2


def nlml_grad(xs, y, sf2, kernel, sn2=0.0, jitter=0.0):
    """(NLML, gradient) in theta = (log sigma_f2, log ell_1..d) with sigma_n2 and the jitter held fixed.

    dNLML/dtheta = 1/2 tr(W dK/dtheta), W = K^-1 - alpha alpha^T, where only the kernel term depends on theta:
      dK_ij/dlog sigma_f2 = sigma_f2 k0(r_ij)                (the noise and jitter on the diagonal do not scale),
      dK_ij/dlog ell_t    = sigma_f2 dk(r_ij) (xs_it - xs_jt)^2   (r^2 = sum_t (x_t / ell_t)^2 differences)."""
    P, s = _mp_rows(xs), _F(sf2)
    n, d = len(P), len(P[0])
    K = kernel_matrix(xs, sf2, kernel, sn2, jitter)
    L = cholesky(K)
    X = tri_inv(L)
    yv = [_F(float(v)) for v in np.asarray(y, np.float64)]
    t = forward(L, yv)
    a = backward_t(L, t)
    f = mp.fdot(t, t) / 2 + mp.fsum(mp.log(L[i][i]) for i in range(n)) + n * mp.log(2 * mp.pi) / 2
    cols = [[X[k][c] for k in range(c, n)] for c in range(n)]      # column c of L^-1 from row c down
    g = [_F(0)] * (d + 1)
    for i in range(n):
        for j in range(i + 1):
            kinv = mp.fdot(cols[i][i - i:], cols[j][i - j:])         # (L^-T L^-1)_ij = sum_{k >= i} X_ki X_kj
            w = kinv - a[i] * a[j]
            if i != j:
                w *= 2                                                # W_ij + W_ji
            df2 = _diff2(P[i], P[j])
            k0, dk = _k0_dk(mp.fsum(df2), kernel)
            g[0] += w * s * k0
            c = w * s * dk
            for q in range(d):
                g[1 + q] += c * df2[q]
    return f, [v / 2 for v in g]


def joint_sigma(xs_train, xs_cand, sf2, kernel, diag_train):
    """Sigma = K** - K*^T (K + diag_train I)^-1 K* over the candidates (no diagonal added: the caller adds diag_add)."""
    K = kernel_matrix(xs_train, sf2, kernel, diag_train, 0.0)
    L = cholesky(K)
    Ks = cross_kernel(xs_train, xs_cand, sf2, kernel)        # (n, m)
    n, m = len(Ks), len(Ks[0])
    V = [forward(L, [Ks[i][c] for i in range(n)]) for c in range(m)]   # V[c] = L^-1 K*[:, c]
    Kss = kernel_matrix(xs_cand, sf2, kernel)
    return [[Kss[a][b] - mp.fdot(V[a], V[b]) for b in range(m)] for a in range(m)]


def joint_mean(xs_train, y, xs_cand, sf2, kernel, diag_train):
    """mu = K*^T alpha."""
    K = kernel_matrix(xs_train, sf2, kernel, diag_train, 0.0)
    a = alpha(cholesky(K), y)
    Ks = cross_kernel(xs_train, xs_cand, sf2, kernel)
    return [mp.fdot([Ks[i][c] for i in range(len(Ks))], a) for c in range(len(Ks[0]))]


def cond2(M):
    """kappa_2 of a symmetric positive definite matrix (list of rows of mpf) from float64 eigenvalues of its rounding:
    the eigenvalues of the rounded matrix are within ~u |M| of the exact ones, so this is accurate to a few digits while
    kappa <~ 1e12 (asserted)."""
    w = np.linalg.eigvalsh(to_np(M))
    k = float(w[-1] / w[0]) if w[0] > 0 else np.inf
    assert 0 < k <= 1e12, f"kappa {k:.3g}: outside the range float64 eigenvalues resolve"
    return k
