"""The FP64 factorisations under every posterior at their block, size and conditioning edges: the K3 refresh (L, L^-1,
alpha and the fast path's operand planes), the likelihood gradient of the device fit and the joint posterior samples.

Every tolerance is an error bound in n, u = 2^-53, a condition number and a stated constant, never a fit to the
observed error.  The standard results used (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed.):
  * a Cholesky factor with backward error dK satisfies |L L^T - K| <= gamma |L| |L|^T, gamma = c n u, and its forward
    error is at most kappa_2(K) times the relative backward error;
  * K3 solves the panels and builds L^-1 with the explicitly inverted 64 x 64 diagonal blocks, which multiplies both
    componentwise bounds by kappa_blk = max_k || |L_kk^-1| |L_kk| ||_inf (Skeel's condition number of a diagonal block,
    taken from the device's own factor);
  * X = L^-1 by column-wise substitution satisfies the right residual bound |L X - I| <= gamma |L| |X|; the left one
    follows from X L - I = L^-1 (L X - I) L, i.e. |X L - I| <= gamma |X| |L| |X| |L|;
  * a perturbation of relative size e in K moves L by kappa e and L^-1 = X by kappa e kappa(L) = kappa^1.5 e, because
    dX = -X dL X and kappa_2(L) = kappa_2(K)^1/2.
The worst error-to-bound ratio of each group, and the range of ratios of every check over its cases, is printed at
the end of the module (pytest -s)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi  # noqa: E402
from optimobo_b200.gp import _KERNELS, current_stream_ptr  # noqa: E402
from oracle import oracle as O  # noqa: E402

import linalg_mpmath as R  # noqa: E402

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
NB = 64
WORST = {}


def _record(group, check, err, bound):
    """Asserts err <= bound and keeps the largest and smallest ratio of each check over its cases (a smallest ratio far
    below 1 shows a case whose bound does not constrain the kernel)."""
    err, bound = float(err), float(bound)
    assert err <= bound, f"group {group} ({check}): error {err:.3e} exceeds its bound {bound:.3e}"
    r = err / bound if bound > 0 else 0.0
    lo, hi = WORST.get((group, check), (np.inf, 0.0))
    WORST[(group, check)] = (min(lo, r), max(hi, r))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        groups = sorted({g for g, _ in WORST})
        print("\nworst error / bound per group: "
              + ", ".join(f"{g} {max(v[1] for (h, _), v in WORST.items() if h == g):.3g}" for g in groups))
        for (g, c), (lo, hi) in sorted(WORST.items()):
            print(f"  {g} {c}: ratio over its cases {lo:.3g} .. {hi:.3g}")


def _okern(kernel):
    return O.KERNEL_MATERN52 if kernel == "matern52" else O.KERNEL_RBF


def _problem(n, d, seed, lo=0.0, hi=1.0):
    rng = np.random.default_rng(seed)
    X = lo + (hi - lo) * rng.random((n, d))
    y = np.sin(3 * X[:, 0]) + X[:, -1] ** 2 + 0.1 * rng.standard_normal(n)
    return X, y


def _gp(X, y, ell, sf2, kernel="matern52", sn2=0.0, jitter=0.0):
    return ob.GPModel(X, y, np.broadcast_to(ell, (X.shape[1],)), sf2, noise=sn2, jitter=jitter, kernel=kernel,
                      device=DEV, max_jitter_tries=0)


def _full(gp, field, dtype, count=None):
    np_ = gp.n_pad
    shape = {_cabi.FIELD_L: (np_, np_), _cabi.FIELD_LINV: (np_, np_), _cabi.FIELD_ALPHA: (np_,),
             _cabi.FIELD_BHI: (np_ * np_,), _cabi.FIELD_BLO: (np_ * np_,), _cabi.FIELD_XS32: (32 * np_,),
             _cabi.FIELD_ALPHA32: (np_,), _cabi.FIELD_STATUS: (4,)}[field]
    return gp._field(field, dtype, shape).cpu().numpy().copy()


def _status(gp):
    return _full(gp, _cabi.FIELD_STATUS, torch.int32)


def _block_cond(L, n):
    """kappa_blk: max over the 64 x 64 diagonal blocks of the device's factor of || |L_kk^-1| |L_kk| ||_inf."""
    worst = 1.0
    for k0 in range(0, n, NB):
        B = np.tril(L[k0:k0 + NB, k0:k0 + NB])
        Bi = np.linalg.inv(B)
        worst = max(worst, np.abs(Bi).dot(np.abs(B)).sum(1).max())
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# a. refresh against mpmath
# ---------------------------------------------------------------------------------------------------------------------
# (n, d, kernel, sigma_f2, sigma_n2 / sigma_f2, ell): n at and around the 64-row block edges, kappa from 1 to 2e10
REFRESH_CASES = [
    (1, 1, "matern52", 1.0, 0.0, 0.5), (2, 5, "rbf", 1e-3, 0.0, 0.7), (63, 12, "matern52", 1.0, 1e-2, 1.0),
    (64, 13, "rbf", 1e3, 0.0, 1.5), (65, 32, "matern52", 1e3, 1e-2, 2.0), (127, 5, "rbf", 1.0, 1e-2, 0.6),
    (128, 1, "matern52", 1e-3, 1e-2, 0.2), (129, 12, "rbf", 1e-3, 0.0, 1.0),
    (129, 1, "matern52", 1.0, 0.0, 0.05),                # noise-free, kappa ~ 2e10
    (64, 32, "rbf", 1.0, 0.0, 3.0), (65, 13, "matern52", 1e-3, 0.0, 0.8), (127, 32, "matern52", 1.0, 0.0, 1.5),
    (128, 5, "rbf", 1e3, 1e-2, 0.5), (2, 1, "rbf", 1e3, 1e-2, 0.3), (63, 1, "rbf", 1.0, 0.0, 0.008),
    (129, 13, "matern52", 1.0, 1e-2, 1.0),
]
C_REFRESH = 8       # e_K = C n u: the device's K (about ten roundings per entry) and the Cholesky's backward error


def _inverse_bounds(Ld, Xd, y, kappa, kinv, e):
    """Error bounds of K^-1 = X^T X and alpha = X^T (X y) as the device forms them from its own L and X = L^-1, all
    linear in kappa:
      * L L^T = K + dK with ||dK|| <= e ||K|| (e = C n u, the relative backward error), so ||(L L^T)^-1 - K^-1|| <=
        kappa e ||K^-1|| -- X^T X depends on L only through L L^T, so the kappa^1.5 of X itself cancels;
      * X - L^-1 = L^-1 (L X - I), |L X - I| <= gamma kappa_blk |L||X| (group b), so ||X - L^-1||_2 <= F =
        gamma kappa_blk || |X||L||X| ||_2 with gamma = e;
      * the two matrix-vector products (k_trmv_lower, k_trmv_lower_t) round by at most n u |X|^T |X| |y|.
    Returns (F, bound on ||X^T X - K^-1||_2, bound on ||alpha - K^-1 y||_2)."""
    n = len(Ld)
    aL, aX = np.abs(Ld), np.abs(Xd)
    F = e * _block_cond(Ld, n) * np.linalg.norm(aX @ aL @ aX, 2)
    xn = np.linalg.norm(Xd, 2)
    d_kinv = kappa * e * kinv + 2 * xn * F + n * U * np.linalg.norm(aX.T @ aX, 2)
    d_alpha = d_kinv * np.linalg.norm(y) + 2 * n * U * np.linalg.norm(aX.T @ (aX @ np.abs(y)))
    return F, d_kinv, d_alpha


@pytest.mark.parametrize("n,d,kernel,sf2,nrel,ell", REFRESH_CASES)
def test_refresh_forward_error_vs_mpmath(n, d, kernel, sf2, nrel, ell):
    """Against the reference factors of K, e = 8 n u:
      ||L - L_ref||_F / ||L_ref||_F <= e kappa,
      ||X - X_ref||_F / ||X_ref||_F <= e kappa^1.5 (the worst case: dX = -X dL X; loose once kappa is large),
      ||alpha - alpha_ref|| <= the kappa-linear bound of _inverse_bounds.
    And against the exact inverse of the device's own L (mpmath from its float64 entries), which isolates the
    triangular inverse at every kappa: ||X - L^-1||_F <= gamma kappa_blk || |L^-1||L||X| ||_F."""
    X, y = _problem(n, d, 1000 + n + d)
    ellv = np.full(d, ell)
    sn2 = nrel * sf2
    gp = _gp(X, y, ellv, sf2, kernel, sn2, 0.0)
    K, L, Xi, a = R.factor(X / ellv, y, sf2, kernel, sn2, 0.0)
    kappa = R.cond2(K)
    Lr, Xr, ar = R.to_np(L), R.to_np(Xi), R.to_np(a)
    e = C_REFRESH * n * U
    Ld, Xd, ad = gp.L.cpu().numpy(), gp.Linv.cpu().numpy(), gp.alpha.cpu().numpy()
    _record("a", "L vs mpmath", np.linalg.norm(Ld - Lr) / np.linalg.norm(Lr), e * kappa)
    _record("a", "L^-1 vs mpmath", np.linalg.norm(Xd - Xr) / np.linalg.norm(Xr), e * kappa ** 1.5)
    kinv = np.linalg.norm(Xr, 2) ** 2
    _, _, d_alpha = _inverse_bounds(Ld, Xd, y, kappa, kinv, e)
    _record("a", "alpha vs mpmath", np.linalg.norm(ad - ar), d_alpha)
    Xown = R.to_np(R.tri_inv(R._mp_rows(Ld)))
    own_bound = e * _block_cond(Ld, n) * np.linalg.norm(np.abs(Xown) @ np.abs(Ld) @ np.abs(Xd))
    _record("a", "L^-1 vs inverse of own L", np.linalg.norm(Xd - Xown), own_bound)
    assert _status(gp)[0] == 0


def test_refresh_covers_an_ill_conditioned_noise_free_case():
    n, d, kernel, sf2, nrel, ell = REFRESH_CASES[8]
    X, _ = _problem(n, d, 1000 + n + d)
    assert nrel == 0.0 and R.cond2(R.kernel_matrix(X / ell, sf2, kernel)) >= 1e8


# ---------------------------------------------------------------------------------------------------------------------
# b. backward error over the whole n range
# ---------------------------------------------------------------------------------------------------------------------
BIG_N = [191, 193, 255, 257, 511, 513, 1023, 1025, 2047, 2049, 4095, 4097, 8191, 8192]
C_BACK = 4


def _K_device(X, ell, sf2, kernel, diag):
    """K in torch FP64 on the device (direct differences), for the sizes where the host would be slow."""
    xs = torch.as_tensor(X / ell, device=DEV)
    r2 = torch.zeros((len(X), len(X)), dtype=torch.float64, device=DEV)
    for t in range(xs.shape[1]):
        r2 += (xs[:, t, None] - xs[None, :, t]) ** 2
    if kernel == "matern52":
        r = torch.sqrt(r2)
        K = sf2 * (1.0 + np.sqrt(5.0) * r + (5.0 / 3.0) * r2) * torch.exp(-np.sqrt(5.0) * r)
    else:
        K = sf2 * torch.exp(-0.5 * r2)
    return K + diag * torch.eye(len(X), dtype=torch.float64, device=DEV)


@pytest.mark.parametrize("i,n", list(enumerate(BIG_N)))
def test_refresh_backward_error_all_sizes(i, n):
    """Residuals of the device's own factors, computed with cuBLAS FP64 matrix products (an implementation independent
    of the kernels under test; their own rounding is covered by the same gamma):
      |L L^T - K| <= gamma kappa_blk |L||L|^T,  |L X - I| <= gamma kappa_blk |L||X|,
      |X L - I| <= gamma kappa_blk |X||L||X||L|,  ||K alpha - y||_inf <= gamma kappa_inf(L) ||K||_inf ||alpha||_inf,
    gamma = 4 n u; K from the float64 oracle on the host up to n = 2049, from torch on the device above.  L^-1 is
    exactly zero above the diagonal and in the padding, and the status word is 0."""
    d = (1, 7, 12, 13, 32)[i % 5]
    kernel = "matern52" if i % 2 == 0 else "rbf"
    X, y = _problem(n, d, n)
    ell = np.full(d, 0.3 * np.sqrt(d))
    sf2, sn2 = 1.5, 1.5e-2
    gp = _gp(X, y, ell, sf2, kernel, sn2, 0.0)
    st = _status(gp)
    assert st[0] == 0
    Lf = gp._field(_cabi.FIELD_L, torch.float64, (gp.n_pad, gp.n_pad))
    Xf = gp._field(_cabi.FIELD_LINV, torch.float64, (gp.n_pad, gp.n_pad))
    assert torch.count_nonzero(torch.triu(Xf, 1)) == 0
    assert torch.count_nonzero(Xf[n:]) == 0 and torch.count_nonzero(Xf[:, n:]) == 0
    L = torch.tril(Lf[:n, :n])
    Xi = Xf[:n, :n].clone()
    if n <= 2049:
        K = torch.as_tensor(O.k_of_r(O.scaled_dist(X, X, ell, "direct"), sf2, _okern(kernel)) + sn2 * np.eye(n),
                            device=DEV)
    else:
        K = _K_device(X, ell, sf2, kernel, sn2)
    kb = _block_cond(L.cpu().numpy(), n)
    g = C_BACK * n * U * kb
    aL, aX = L.abs(), Xi.abs()
    eye = torch.eye(n, dtype=torch.float64, device=DEV)
    tiny = 1e-300
    r = ((L @ L.T - K).abs() / (g * (aL @ aL.T) + tiny)).max().item()
    _record("b", "|LL^T - K|", r, 1.0)
    r = ((L @ Xi - eye).abs() / (g * (aL @ aX) + tiny)).max().item()
    _record("b", "|LX - I|", r, 1.0)
    M = aX @ aL
    r = ((Xi @ L - eye).abs() / (g * (M @ M) + tiny)).max().item()
    _record("b", "|XL - I|", r, 1.0)
    del M
    a = gp.alpha
    yt = torch.as_tensor(y, device=DEV)
    inf = lambda A: A.abs().sum(1).max().item()  # noqa: E731
    kappa_L = inf(L) * inf(Xi)
    res = (K @ a - yt).abs().max().item()
    _record("b", "K alpha - y", res, C_BACK * n * U * kappa_L * inf(K) * a.abs().max().item())


# ---------------------------------------------------------------------------------------------------------------------
# c. exact scaling
# ---------------------------------------------------------------------------------------------------------------------
def _planes(gp):
    return (_full(gp, _cabi.FIELD_BHI, torch.int16).view(np.uint16), _full(gp, _cabi.FIELD_BLO, torch.int16).view(np.uint16),
            _full(gp, _cabi.FIELD_ALPHA32, torch.float32), _full(gp, _cabi.FIELD_XS32, torch.float32))


def _bf16_value(bits):
    return (bits.astype(np.uint32) << 16).view(np.float32)


# (n, d, kernel, sn2 / sf2, ell, expected plane format)
SCALING_CASES = [(200, 5, "matern52", 2e-2, 0.7, "f8c"), (150, 3, "rbf", 0.0, 0.5, "fp16x3"),
                 (130, 20, "matern52", 2e-2, 1.2, "bf16x3")]


@pytest.mark.parametrize("n,d,kernel,nrel,ell,fmt", SCALING_CASES)
@pytest.mark.parametrize("k", [-8, 8])
def test_power_of_two_scaling_is_exact(n, d, kernel, nrel, ell, fmt, k):
    """sigma_f2, sigma_n2 and the jitter times 4^k: L scales by 2^k, L^-1 by 2^-k and alpha by 4^-k exactly; the f8c
    and fp16 planes and ALPHA32 are bit-identical (the power-of-two plane scale absorbs 2^k), the bf16 planes scale by
    2^k; the joint-sample factor scales by 2^k and the mean is unchanged.  X and ell times 2^k: everything identical,
    XS32 included.  Every step is homogeneous and sqrt(4 p) = 2 sqrt(p), so any difference is a hidden constant."""
    X, y = _problem(n, d, 77 + n)
    sf2, jit = 0.8, 1e-9
    sn2 = nrel * sf2
    s4, s2 = 4.0 ** k, 2.0 ** k
    a = _gp(X, y, ell, sf2, kernel, sn2, jit)
    b = _gp(X, y, ell, sf2 * s4, kernel, sn2 * s4, jit * s4)
    c = _gp(X * s2, y, ell * s2, sf2, kernel, sn2, jit)
    assert a.plane_format == b.plane_format == c.plane_format == fmt
    La, Lb = a.L.cpu().numpy(), b.L.cpu().numpy()
    assert np.array_equal(Lb, La * s2)
    assert np.array_equal(b.Linv.cpu().numpy(), a.Linv.cpu().numpy() / s2)
    assert np.array_equal(b.alpha.cpu().numpy(), a.alpha.cpu().numpy() / s4)
    pa, pb, pc = _planes(a), _planes(b), _planes(c)
    if fmt == "bf16x3":
        for q in (0, 1):
            assert np.array_equal(_bf16_value(pb[q]), _bf16_value(pa[q]) * np.float32(s2))
    else:
        assert np.array_equal(pa[0], pb[0]) and np.array_equal(pa[1], pb[1])
    assert np.array_equal(pa[2], pb[2])
    for f in (_cabi.FIELD_L, _cabi.FIELD_LINV):
        assert np.array_equal(np.tril(_full(a, f, torch.float64)), np.tril(_full(c, f, torch.float64)))
    assert np.array_equal(a.alpha.cpu().numpy(), c.alpha.cpu().numpy())
    for q in range(4):
        assert np.array_equal(pa[q], pc[q])
    # joint samples: y = 0 makes mu = 0, so out is the factor itself (Z = I)
    m = 70
    Xc = np.random.default_rng(5).random((m, d))
    a0, b0 = _gp(X, 0 * y, ell, sf2, kernel, sn2, jit), _gp(X, 0 * y, ell, sf2 * s4, kernel, sn2 * s4, jit * s4)
    Fa = a0.posterior_samples_from(Xc, np.eye(m), jitter=1e-6 * sf2, max_jitter_tries=0)[:, 0, :]
    Fb = b0.posterior_samples_from(Xc, np.eye(m), jitter=1e-6 * sf2 * s4, max_jitter_tries=0)[:, 0, :]
    assert np.array_equal(Fb, Fa * s2) and np.count_nonzero(np.diag(Fa)) == m
    ma = a.posterior_samples_from(Xc, np.zeros((m, 2)), jitter=1e-6 * sf2, max_jitter_tries=0)
    mb = b.posterior_samples_from(Xc, np.zeros((m, 2)), jitter=1e-6 * sf2 * s4, max_jitter_tries=0)
    assert np.array_equal(ma, mb)


# ---------------------------------------------------------------------------------------------------------------------
# d. reproducibility
# ---------------------------------------------------------------------------------------------------------------------
def test_refresh_is_bit_reproducible_at_max_n():
    n, d = 8192, 6
    X, y = _problem(n, d, 3)
    gp = _gp(X, y, np.full(d, 0.5), 1.0, "matern52", 1e-2, 0.0)
    fields = (_cabi.FIELD_L, _cabi.FIELD_LINV, _cabi.FIELD_ALPHA, _cabi.FIELD_BHI, _cabi.FIELD_BLO,
              _cabi.FIELD_ALPHA32, _cabi.FIELD_XS32)
    # state_field counts elements of each field's own type: 8 bytes for L / L^-1 / alpha, 2 for the 16-bit planes
    # (the f8c lo field holds two n_pad^2 byte planes in the same space), 4 for ALPHA32 / XS32
    esize = {_cabi.FIELD_L: 8, _cabi.FIELD_LINV: 8, _cabi.FIELD_ALPHA: 8, _cabi.FIELD_BHI: 2, _cabi.FIELD_BLO: 2,
             _cabi.FIELD_ALPHA32: 4, _cabi.FIELD_XS32: 4}

    def raw(f):
        off, cnt = _cabi.state_field(n, d, f)
        return gp.state[off:off + cnt * esize[f]]

    assert raw(_cabi.FIELD_L).numel() == gp.n_pad ** 2 * 8 and raw(_cabi.FIELD_BLO).numel() == 2 * gp.n_pad ** 2
    first = [raw(f).clone() for f in fields]
    gp.refresh()
    for f, v in zip(fields, first):
        assert torch.equal(raw(f), v), f


# ---------------------------------------------------------------------------------------------------------------------
# e. operand planes, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
def _e4m3(x32):
    """float32 -> e4m3 byte with __NV_SATFINITE: torch's cast turns overflow into NaN, so clamp to +-448 first."""
    t = torch.from_numpy(np.ascontiguousarray(x32)).clamp(-448.0, 448.0)
    return t.to(torch.float8_e4m3fn).view(torch.uint8).numpy()


def _bf16_bits(x32):
    return torch.from_numpy(np.ascontiguousarray(x32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def _expected_format(gp, kappa_limit, allow_f8c):
    dg = np.diag(_full(gp, _cabi.FIELD_L, torch.float64))[: gp.n]
    ratio = dg.max() / dg.min()
    kappa = ratio * ratio
    if allow_f8c and gp.d <= 12 and kappa <= kappa_limit:
        return "f8c"
    return "fp16x3" if kappa > 100.0 else "bf16x3"


def _check_planes(gp, kappa_limit=100.0, allow_f8c=True):
    """Re-encodes the device's own L^-1 on the host as k_absmax_lower / k_finalize / k_publish_scale do and compares
    every bit; returns the plane format."""
    n, np_, sf2 = gp.n, gp.n_pad, gp.variance
    fmt = _expected_format(gp, kappa_limit, allow_f8c)
    assert gp.plane_format == fmt
    Xf = _full(gp, _cabi.FIELD_LINV, torch.float64)
    valid = np.tril(np.ones((np_, np_), bool))
    valid[n:] = False
    valid[:, n:] = False
    assert np.count_nonzero(Xf[~valid]) == 0
    mx = np.abs(Xf[valid]).max() * sf2
    if fmt == "bf16x3":
        sc = 1.0
    else:
        q = np.log2(16384.0 / mx)
        assert abs(q - np.round(q)) > 1e-9, "16384 / max is within an ulp of a power of two: pick other inputs"
        sc = 2.0 ** np.floor(q)
    t = (Xf * sf2 * sc).reshape(-1)
    bhi = _full(gp, _cabi.FIELD_BHI, torch.int16).view(np.uint16)
    blo = _full(gp, _cabi.FIELD_BLO, torch.int16).view(np.uint16)
    if fmt == "bf16x3":
        h = _bf16_bits(t.astype(np.float32))
        lo = _bf16_bits((t - _bf16_value(h).astype(np.float64)).astype(np.float32))
        assert np.array_equal(bhi, h) and np.array_equal(blo, lo)
    else:
        h = t.astype(np.float32).astype(np.float16)
        assert np.array_equal(bhi, h.view(np.uint16))
        r = (t - h.astype(np.float64)).astype(np.float32)
        if fmt == "fp16x3":
            assert np.array_equal(blo, r.astype(np.float16).view(np.uint16))
        else:
            c = blo.view(np.uint8)
            assert np.array_equal(c[: np_ * np_], _e4m3((t * (1.0 / 4096.0)).astype(np.float32)))
            assert np.array_equal(c[np_ * np_:], _e4m3(r))
    # zero outside the valid lower triangle (each f8c lo plane on its own)
    lo_planes = (blo.view(np.uint8)[: np_ * np_], blo.view(np.uint8)[np_ * np_:]) if fmt == "f8c" else (blo,)
    for p in (bhi,) + lo_planes:
        assert np.count_nonzero(p.reshape(np_, np_)[~valid]) == 0
    al = _full(gp, _cabi.FIELD_ALPHA, torch.float64)
    assert np.array_equal(_full(gp, _cabi.FIELD_ALPHA32, torch.float32), (al * sf2).astype(np.float32))
    return fmt


# (n, d, kernel, sf2, sn2 / sf2, ell, expected format)
PLANE_CASES = [(300, 7, "matern52", 2.5, 2e-2, 0.6, "f8c"), (129, 12, "rbf", 0.3, 3e-2, 0.9, "f8c"),
               (257, 4, "matern52", 1.7, 0.0, 0.4, "fp16x3"), (64, 3, "rbf", 3.0, 1e-4, 0.5, "fp16x3"),
               (200, 13, "matern52", 0.9, 2e-2, 1.5, "bf16x3"), (65, 32, "rbf", 1.3, 3e-2, 3.0, "bf16x3")]


@pytest.mark.parametrize("n,d,kernel,sf2,nrel,ell,fmt", PLANE_CASES)
def test_operand_planes_bit_exact(n, d, kernel, sf2, nrel, ell, fmt):
    X, y = _problem(n, d, 31 + n)
    gp = _gp(X, y, ell, sf2, kernel, nrel * sf2, 1e-9)
    assert _check_planes(gp) == fmt


def _planes_in_fresh_process(env, cases):
    code = (f"import sys\nsys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
            f"import test_gpu_linalg_edges as T\nT._planes_cases({cases!r}, {env!r})\n")
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]


def _planes_cases(cases, env):
    kappa_limit = float(env.get("OMBO_F8C_KAPPA", 100.0))
    allow = "OMBO_NO_F8C" not in env
    for (n, d, kernel, sf2, nrel, ell, fmt) in cases:
        X, y = _problem(n, d, 31 + n)
        gp = _gp(X, y, ell, sf2, kernel, nrel * sf2, 1e-9)
        assert _check_planes(gp, kappa_limit, allow) == fmt, (n, d, fmt)


def test_operand_planes_without_f8c_and_with_a_raised_kappa_limit():
    """OMBO_NO_F8C: the well-conditioned d <= 12 GPs get bf16 x3 planes; OMBO_F8C_KAPPA = 1e7: the fp16 cases
    (kappa > 100, d <= 12) get f8c planes instead.  Both read once per process, so each runs in a fresh one."""
    _planes_in_fresh_process({"OMBO_NO_F8C": "1"}, [c[:6] + ("bf16x3",) for c in PLANE_CASES[:2]] + [PLANE_CASES[2]])
    _planes_in_fresh_process({"OMBO_F8C_KAPPA": "1e7"}, [c[:6] + ("f8c",) for c in PLANE_CASES[2:4]])


# ---------------------------------------------------------------------------------------------------------------------
# f. likelihood and gradient
# ---------------------------------------------------------------------------------------------------------------------
def _nlml_device(X, y, ell, sf2, kernel, sn2, jitter, state=None):
    """ombo_gp_nlml_grad -> (rc, [NLML, gradient], state blob holding the L and L^-1 it used)."""
    n, d = X.shape
    dev = torch.device(DEV)
    Xd, yd = torch.as_tensor(X, device=dev).contiguous(), torch.as_tensor(y, device=dev).contiguous()
    if state is None:
        state = torch.empty(_cabi.state_bytes(n, d), dtype=torch.uint8, device=dev)
    ellc = (C.c_double * d)(*np.broadcast_to(ell, (d,)).tolist())
    spec = _cabi.GpSpec(n=n, d=d, kernel=_KERNELS[kernel], reserved=0, sigma_f2=float(sf2), sigma_n2=float(sn2),
                        jitter=float(jitter), X=Xd.data_ptr(), y=yd.data_ptr(), ell=ellc)
    out = (C.c_double * (d + 2))()
    rc = _cabi.lib().ombo_gp_nlml_grad(_cabi.Context.get(0).handle, C.byref(spec), C.c_void_p(state.data_ptr()), out,
                                       current_stream_ptr(dev))
    return rc, np.frombuffer(out, dtype=np.float64, count=d + 2).copy(), state


def _state_matrix(state, n, d, field):
    np_ = _cabi.lib().ombo_n_pad(n)
    off, cnt = _cabi.state_field(n, d, field)
    return state[off:off + cnt * 8].view(torch.float64).view(np_, np_)[:n, :n].cpu().numpy()


# (n, d, kernel, sn2 / sf2, ell)
NLML_CASES = [(1, 1, "matern52", 0.0, 0.5), (2, 2, "rbf", 1e-2, 0.6), (15, 12, "matern52", 1e-2, 1.0),
              (16, 13, "rbf", 0.0, 1.2), (17, 32, "matern52", 0.0, 2.0), (64, 2, "rbf", 1e-2, 0.3),
              (65, 12, "matern52", 1e-2, 0.9), (129, 1, "rbf", 1e-2, 0.05), (129, 5, "matern52", 0.0, 0.6),
              (17, 1, "matern52", 1e-2, 0.2), (64, 32, "matern52", 1e-2, 2.5), (65, 13, "rbf", 0.0, 1.4)]
C_NLML = 8


@pytest.mark.parametrize("n,d,kernel,nrel,ell", NLML_CASES)
def test_nlml_and_gradient_vs_mpmath(n, d, kernel, nrel, ell):
    """With dKinv, dalpha the kappa-linear bounds of _inverse_bounds (e = 8 n u) from the device's own L and L^-1:
      |f - f_ref| <= 1/2 ||y|| dalpha + 1/2 n kappa e (log det: tr(K^-1 dK)) + (n + 2) u (sum of |terms| of f),
      |g_k - g_ref_k| <= 1/2 sqrt(n) (dKinv + 2 ||alpha|| dalpha) ||dK/dtheta_k||_F (W = K^-1 - alpha alpha^T)
                         + n u 1/2 sum_ij |W_ij dK_ij/dtheta_k| (the rounding of the reduction itself).
    The sigma_n2 > 0 cases check the noise term, which the gradient in sigma_f2 must leave out."""
    X, y = _problem(n, d, 500 + n + d)
    sf2 = 1.3
    ellv = np.full(d, ell)
    sn2 = nrel * sf2
    rc, v, state = _nlml_device(X, y, ellv, sf2, kernel, sn2, 0.0)
    _cabi.check(rc)
    Ld = np.tril(_state_matrix(state, n, d, _cabi.FIELD_L))
    Xd = _state_matrix(state, n, d, _cabi.FIELD_LINV)
    xs = X / ellv
    f, g = R.nlml_grad(xs, y, sf2, kernel, sn2, 0.0)
    K = R.kernel_matrix(xs, sf2, kernel, sn2, 0.0)
    kappa = R.cond2(K)
    Kf = R.to_np(K)
    kinv = 1.0 / np.linalg.eigvalsh(Kf)[0]
    e = C_NLML * n * U
    _, d_kinv, d_alpha = _inverse_bounds(Ld, Xd, y, kappa, kinv, e)
    Lr = np.linalg.cholesky(Kf)
    ar = np.linalg.solve(Kf, y)
    f_terms = abs(0.5 * y @ ar) + np.abs(np.log(np.diag(Lr))).sum() + 0.5 * n * np.log(2 * np.pi)
    _record("f", "NLML vs mpmath", abs(v[0] - float(f)),
            0.5 * np.linalg.norm(y) * d_alpha + 0.5 * n * kappa * e + (n + 2) * U * f_terms)
    W = np.linalg.inv(Kf) - np.outer(ar, ar)
    d_w = d_kinv + 2 * np.linalg.norm(ar) * d_alpha
    k0 = Kf - sn2 * np.eye(n)
    diff2 = (xs[:, None, :] - xs[None, :, :]) ** 2
    r2 = diff2.sum(-1)
    if kernel == "matern52":
        r = np.sqrt(r2)
        dk = sf2 * (5.0 / 3.0) * (1 + np.sqrt(5.0) * r) * np.exp(-np.sqrt(5.0) * r)
    else:
        dk = k0
    dK = [k0] + [dk * diff2[:, :, t] for t in range(d)]
    gr = R.to_np(g)
    for q in range(d + 1):
        bound = 0.5 * np.sqrt(n) * d_w * np.linalg.norm(dK[q]) + n * U * 0.5 * np.abs(W * dK[q]).sum()
        _record("f", "gradient vs mpmath", abs(v[1 + q] - gr[q]), bound + 1e-300)


@pytest.mark.parametrize("n,d", [(1025, 3), (2049, 2), (4096, 4), (8192, 2)])
def test_gradient_vs_central_differences_large_n(n, d):
    """The device's gradient against central differences (h = 1e-4) of the device's own NLML, sigma_n2 = 1e-2 (well
    conditioned): truncation ~h^2 |f'''| and rounding ~u kappa |f| / h stay far below 1e-4 max|g|.  This catches the
    systematic faults of the (n/16)^2-block reduction at these sizes (a dropped or doubled row or column of partial
    blocks, a wrong stride, a missing or extra term) but not necessarily one lost block: at n = 8192 a single block of
    262144 carries ~4e-6 of the sum unless cancellation makes it larger.  The mpmath comparison above holds the
    reduction to its rounding bound at n <= 129."""
    X, y = _problem(n, d, n)
    ell, sf2, sn2 = np.full(d, 0.4), 1.0, 1e-2
    theta = np.log(np.concatenate(([sf2], ell)))
    state = torch.empty(_cabi.state_bytes(n, d), dtype=torch.uint8, device=DEV)

    def f(th):
        rc, v, _ = _nlml_device(X, y, np.exp(th[1:]), np.exp(th[0]), "matern52", sn2, 0.0, state)
        _cabi.check(rc)
        return v

    v = f(theta)
    g = v[1:]
    h = 1e-4
    fd = np.empty(d + 1)
    for q in range(d + 1):
        e = np.zeros(d + 1)
        e[q] = h
        fd[q] = (f(theta + e)[0] - f(theta - e)[0]) / (2 * h)
    _record("f", "gradient vs central differences", np.abs(g - fd).max(), 1e-4 * np.abs(g).max())


def test_nlml_not_pd_with_duplicate_rows():
    X = np.array([[0.1, 0.2], [0.3, 0.9], [0.1, 0.2], [0.5, 0.5]])
    rc, _, _ = _nlml_device(X, np.arange(4.0), np.ones(2), 1.0, "matern52", 0.0, 0.0)
    assert rc == _cabi.ERR_NOT_PD


# ---------------------------------------------------------------------------------------------------------------------
# g. joint samples
# ---------------------------------------------------------------------------------------------------------------------
def _factor_of_samples(gp, Xc, diag_jitter, tries=0):
    """Z = I_m with y = 0 (mu = 0): the draws are the factor chol(Sigma + (noise + jitter) I) itself, exactly -- every
    sum above the diagonal holds only exact zeros."""
    m = len(Xc)
    F = gp.posterior_samples_from(Xc, np.eye(m), jitter=diag_jitter, max_jitter_tries=tries)[:, 0, :]
    assert np.count_nonzero(np.triu(F, 1)) == 0
    return F


@pytest.mark.parametrize("n,m,d,kernel", [(1, 1, 2, "matern52"), (64, 2, 3, "rbf"), (129, 63, 5, "matern52"),
                                          (64, 64, 12, "matern52"), (1, 65, 1, "rbf"), (129, 129, 4, "rbf")])
def test_joint_samples_vs_mpmath(n, m, d, kernel):
    """||F - chol(Sigma_ref + diag I)||_F / ||.||_F <= kappa(S) (dS / ||S|| + e_m), with S = Sigma + diag I,
    dS = 2 e kappa(K)^1.5 ||K^-1|| ||K*||^2 + e (||K**|| + ||V||^2) the error of the device's Sigma (e = 8 n u, the
    error of L^-1 as in group a; the second term the cancellation in K** - V V^T) and e_m = 8 m u."""
    X, _ = _problem(n, d, 600 + n + m)
    Xc = np.random.default_rng(m).random((m, d)) * 1.2 - 0.1
    ell, sf2 = np.full(d, 0.5 * np.sqrt(d)), 0.7
    sn2, jit = 1e-3 * sf2, 1e-5 * sf2
    gp = _gp(X, np.zeros(n), ell, sf2, kernel, sn2, 0.0)
    F = _factor_of_samples(gp, Xc, jit)
    S = R.joint_sigma(X / ell, Xc / ell, sf2, kernel, sn2)
    Sd = R.to_np(S) + (sn2 + jit) * np.eye(m)
    import mpmath as mp
    Sm = [[S[i][j] + (mp.mpf(sn2) + mp.mpf(jit) if i == j else 0) for j in range(m)] for i in range(m)]
    Lm = R.to_np(R.cholesky(Sm))
    K = R.kernel_matrix(X / ell, sf2, kernel, sn2, 0.0)
    kK = R.cond2(K)
    kinv = 1.0 / np.linalg.eigvalsh(R.to_np(K))[0]
    Ks = O.k_of_r(O.scaled_dist(X, Xc, ell, "direct"), sf2, _okern(kernel))
    V = np.linalg.solve(np.linalg.cholesky(R.to_np(K)), Ks)
    e = C_REFRESH * n * U
    nS = np.linalg.norm(Sd, 2)
    dS = 2 * e * kK ** 1.5 * kinv * np.linalg.norm(Ks, 2) ** 2 + e * (sf2 * m + np.linalg.norm(V, 2) ** 2)
    kS = R.cond2(Sm)
    _record("g", "factor vs mpmath", np.linalg.norm(F - Lm) / np.linalg.norm(Lm), kS * (dS / nS + 8 * m * U))


def _sigma_products(gp, Xc, F, diag):
    """The backward-error ratio max |F F^T - S| / B of the device's factor F of S = K** - V V^T + diag I, with S formed
    by cuBLAS FP64 from the device's own L^-1 (V = K* X^T) and
    B = gamma_m kappa_blk |F||F|^T + (n + 16) u (|K**| + |V||V|^T + 2 |K*||X|^T|V|^T) (the cancellation in K** - V V^T
    and the rounding of V), gamma_m = 4 m u."""
    m, n = F.shape[0], gp.n
    xs = torch.as_tensor(Xc / gp.lengthscale, device=DEV)
    xt = torch.as_tensor(gp.X.cpu().numpy() / gp.lengthscale, device=DEV)

    def kern(A, B):
        r2 = torch.zeros((len(A), len(B)), dtype=torch.float64, device=DEV)
        for t in range(A.shape[1]):
            r2 += (A[:, t, None] - B[None, :, t]) ** 2
        if gp.kernel_name == "matern52":
            r = torch.sqrt(r2)
            return gp.variance * (1.0 + np.sqrt(5.0) * r + (5.0 / 3.0) * r2) * torch.exp(-np.sqrt(5.0) * r)
        return gp.variance * torch.exp(-0.5 * r2)

    Kss, Ks = kern(xs, xs), kern(xs, xt)                 # (m, m), (m, n)
    Xi = gp.Linv
    V = Ks @ Xi.T
    S = Kss - V @ V.T + diag * torch.eye(m, dtype=torch.float64, device=DEV)
    Ft = torch.as_tensor(F, device=DEV)
    kb = _block_cond(F, m)
    aF, aV = Ft.abs(), V.abs()
    B = 4 * m * U * kb * (aF @ aF.T) + (n + 16) * U * (Kss.abs() + aV @ aV.T + 2 * (Ks.abs() @ Xi.abs().T) @ aV.T)
    return ((Ft @ Ft.T - S).abs() / (B + 1e-300)).max().item()


@pytest.mark.parametrize("m,d", [(127, 3), (191, 5), (193, 8), (1000, 10), (2047, 6), (3200, 32), (4096, 12)])
def test_joint_samples_backward_error(m, d):
    n = 300
    X, _ = _problem(n, d, m)
    gp = _gp(X, np.zeros(n), np.full(d, 0.3 * np.sqrt(d)), 1.1, "matern52", 0.0, 1e-8)
    Xc = np.random.default_rng(m + 1).random((m, d))
    jit = 1e-6 * gp.variance
    F = _factor_of_samples(gp, Xc, jit)
    _record("g", "backward error", _sigma_products(gp, Xc, F, gp.noise + jit), 1.0)


def _turbo_cloud(X, y, ell, length, n_cand, rng):
    """Candidates as TuRBO_1.create_candidates builds them: a Sobol design in the trust region of side `length`
    around the incumbent, each coordinate perturbed with probability min(20 / d, 1)."""
    from scipy.stats import qmc
    d = X.shape[1]
    x_center = X[int(np.argmin(y))][None, :]
    w = ell / ell.mean()
    w = w / np.prod(np.power(w, 1.0 / len(w)))
    lb = np.clip(x_center - w * length / 2.0, 0.0, 1.0)
    ub = np.clip(x_center + w * length / 2.0, 0.0, 1.0)
    sample = qmc.Sobol(d=d, scramble=False).random(n=n_cand)
    sample = qmc.scale(sample, lb[0], np.maximum(ub[0], lb[0] + 1e-12))
    mask = rng.random((n_cand, d)) <= min(20.0 / d, 1.0)
    ind = np.where(mask.sum(1) == 0)[0]
    if len(ind):
        mask[ind, rng.integers(0, max(d - 1, 1), size=len(ind))] = True
    Xc = x_center.copy() * np.ones((n_cand, d))
    Xc[mask] = sample[mask]
    return Xc


@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("d,length", [(10, 0.4), (10, 0.5 ** 7), (32, 0.5 ** 4), (32, 0.5 ** 7)])
def test_joint_samples_turbo_clouds(d, length):
    """TuRBO's Thompson draw on its own candidate cloud (m = 100 d): the backward error holds at the jitter the
    retry settled on, and that jitter follows GPModel.posterior_samples' ladder: 1e-8 sigma_f2, then x10 per
    failure, the rung below it failing (not positive definite)."""
    rng = np.random.default_rng(d)
    n, m = 60, 100 * d
    X = rng.random((n, d))
    y = np.sum((X - 0.4) ** 2, 1)
    ell = rng.uniform(0.3, 1.2, d)
    Xc = _turbo_cloud(X, y, ell, length, m, rng)
    gp = _gp(X, 0 * y, ell, 0.9, "matern52", 0.0, 1e-8)
    F = gp.posterior_samples_from(Xc, np.eye(m), max_jitter_tries=6)[:, 0, :]
    jit = gp.sample_jitter
    rung = np.log10(jit / (1e-8 * gp.variance))
    assert abs(rung - np.round(rung)) < 1e-9 and 0 <= np.round(rung) <= 6
    _record("g", "backward error, TuRBO cloud", _sigma_products(gp, Xc, F, gp.noise + jit), 1.0)
    if np.round(rung) > 0:
        with pytest.raises(_cabi.NotPositiveDefinite):
            gp.posterior_samples_from(Xc, np.zeros((m, 1)), jitter=jit / 10, max_jitter_tries=0)


def test_joint_samples_limits():
    """m = 16384 and S = 4 run, and Z = 0 returns the posterior mean of ob.posterior (FP64): within
    c n u sum_i |K*_ci alpha_i| of it, two summation orders of the same products; m = 16385 or S = 4097 is rejected."""
    n, d = 200, 4
    X, y = _problem(n, d, 9)
    gp = _gp(X, y, np.full(d, 0.5), 1.0, "matern52", 1e-2, 0.0)
    m = 16384
    Xc = np.random.default_rng(10).random((m, d))
    out = gp.posterior_samples_from(Xc, np.zeros((m, 4)), jitter=1e-2, max_jitter_tries=0)[:, 0, :]
    assert np.all(out == out[:, :1])
    mu_ref = ob.posterior([gp], Xc)[0][0].cpu().numpy()
    Ks = O.k_of_r(O.scaled_dist(Xc, X, gp.lengthscale, "direct"), 1.0)
    scale = np.abs(Ks) @ np.abs(gp.alpha.cpu().numpy())
    _record("g", "mean at m = 16384", np.max(np.abs(out[:, 0] - mu_ref) / (4 * n * U * scale)), 1.0)
    with pytest.raises(_cabi.OmboError) as ei:
        gp.posterior_samples_from(np.zeros((m + 1, d)), np.zeros((m + 1, 1)), jitter=1e-2, max_jitter_tries=0)
    assert ei.value.code == _cabi.ERR_INVALID
    with pytest.raises(_cabi.OmboError) as ei:
        gp.posterior_samples_from(Xc[:8], np.zeros((8, 4097)), jitter=1e-2, max_jitter_tries=0)
    assert ei.value.code == _cabi.ERR_INVALID


def test_joint_samples_above_diagonal_equal_mu():
    """With y != 0 and Z = I, out - mu is the factor: the entries above the diagonal equal mu exactly."""
    n, d, m = 90, 3, 77
    X, y = _problem(n, d, 12)
    gp = _gp(X, y, np.full(d, 0.5), 1.0, "rbf", 1e-3, 0.0)
    Xc = np.random.default_rng(13).random((m, d))
    out = gp.posterior_samples_from(Xc, np.eye(m), jitter=1e-6, max_jitter_tries=0)[:, 0, :]
    mu = gp.posterior_samples_from(Xc, np.zeros((m, 1)), jitter=1e-6, max_jitter_tries=0)[:, 0, 0]
    iu = np.triu_indices(m, 1)
    assert np.array_equal(out[iu], mu[iu[0]])
    assert np.all(np.diag(out) != mu)
