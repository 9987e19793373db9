"""CPU: the premises of the Kriging-believer batches (acquisition.propose_batch) on the FP64 oracle, and the spec_for
closures of the two optimisers.

(a) Conditioning a GP on (x1, mu(x1)) leaves the mean unchanged and does not raise any variance (Matern and RBF, with
    and without noise).
(b) After one believer update, EI, the exact 2-D EHVI and the box EHVI of 3 objectives never rise beyond FP64
    rounding, for a believed point the front dominates, one it does not and one beyond the reference point.
(c) The closures: the front grows only by non-dominated believed rows inside the reference point, and the EI incumbent
    and the decomposition's g_min are minima."""
import numpy as np
import pytest

from oracle import oracle as O
from ehvi_oracle import ehvi_grid_batched

import optimobo_b200 as ob
from optimobo_b200 import _cabi, host_prep
from optimobo_b200.algorithms.optimisers import MonoSurrogateOptimiser, MultiSurrogateOptimiser


def _states(X, Y, kernel, noise):
    d = X.shape[1]
    return [O.gp_fit_state(X, Y[:, i], 0.4 * np.ones(d), 1.0 + i, sigma_n2=noise, kernel=kernel)
            for i in range(Y.shape[1])]


def _believe(states, x1):
    """Each state conditioned on its own mean at x1, with the same hyper-parameters."""
    out = []
    for s in states:
        mu1 = O.gp_posterior(s, x1[None, :])[0][0]
        out.append(O.gp_fit_state(np.vstack([s["X"], x1]), np.append(s["y"], mu1), s["ell"], s["sigma_f2"],
                                  sigma_n2=s["sigma_n2"], jitter=s["jitter"], kernel=s["kernel"]))
    return out


def _zdt(X, k=2):
    f1 = X[:, 0]
    g = 1 + 9.0 / (X.shape[1] - 1) * X[:, 1:].sum(1)
    cols = [f1, g * (1 - np.sqrt(f1 / g))]
    if k == 3:
        cols.append(g * (1 - X[:, 1]) + 0.5 * f1)
    return np.column_stack(cols)


@pytest.mark.parametrize("kernel", [O.KERNEL_MATERN52, O.KERNEL_RBF])
@pytest.mark.parametrize("noise", [0.0, 1e-3])
def test_believer_keeps_mean_and_lowers_variance(kernel, noise):
    rng = np.random.default_rng(1)
    X = rng.random((25, 3))
    Y = _zdt(X)
    states = _states(X, Y, kernel, noise)
    Xc = rng.random((2000, 3))
    for x1 in (Xc[0], X[3] + 1e-3, rng.random(3)):
        for s, s1 in zip(states, _believe(states, x1)):
            mu, var = O.gp_posterior(s, Xc)
            mu1, var1 = O.gp_posterior(s1, Xc)
            np.testing.assert_allclose(mu1, mu, rtol=1e-9, atol=1e-9 * np.abs(mu).max())
            assert np.all(var1 <= var * (1 + 1e-9) + 1e-15)


def _three_kinds(pf, r, mu_bel):
    """x1 classes by where the believed objective vector falls: dominated by the front, not dominated, beyond r."""
    dominated = np.array([np.any(np.all(pf <= y, axis=1)) for y in mu_bel])
    beyond = np.any(mu_bel > r, axis=1)
    return {"dominated": np.flatnonzero(dominated & ~beyond), "non_dominated": np.flatnonzero(~dominated & ~beyond),
            "beyond_r": np.flatnonzero(beyond)}


def _front_after(pf, y, r):
    return host_prep.calc_pf(np.vstack([pf, y])) if np.all(y <= r) else pf


def _no_rise(new, old):
    assert np.all(new <= old + 1e-12 * max(np.abs(old).max(), 1e-300) + 1e-300), float(np.max(new - old))


@pytest.mark.parametrize("k", [2, 3])
def test_acquisitions_never_rise_after_a_believer_step(k):
    rng = np.random.default_rng(2)
    X = rng.random((30, 4))
    Y = _zdt(X, k)
    pf = host_prep.calc_pf(Y)
    r = np.quantile(Y, 0.8, axis=0)                     # some believed points fall beyond it
    pf = pf[np.all(pf <= r, axis=1)]
    states = _states(X, Y, O.KERNEL_MATERN52, 0.0)
    Xc = rng.random((400, 4))
    post = [O.gp_posterior(s, Xc) for s in states]
    mu_bel = np.column_stack([p[0] for p in post])
    kinds = _three_kinds(pf, r, mu_bel)
    for name, idx in kinds.items():
        assert len(idx), name
        x1, y1 = Xc[idx[0]], mu_bel[idx[0]]
        post1 = [O.gp_posterior(s, Xc) for s in _believe(states, x1)]
        front1 = _front_after(pf, y1, r)
        mu = np.column_stack([p[0] for p in post]); var = np.column_stack([p[1] for p in post])
        mu1 = np.column_stack([p[0] for p in post1]); var1 = np.column_stack([p[1] for p in post1])
        if k == 2:
            old = O.ehvi_batched(mu[:, 0], mu[:, 1], var[:, 0], var[:, 1], pf, r, None, "exact")
            new = O.ehvi_batched(mu1[:, 0], mu1[:, 1], var1[:, 0], var1[:, 1], front1, r, None, "exact")
            _no_rise(new, old)
            # EI on objective 0 with the believed incumbent
            best = Y[:, 0].min()
            _no_rise(O.expected_improvement(mu1[:, 0], var1[:, 0], min(best, y1[0])),
                     O.expected_improvement(mu[:, 0], var[:, 0], best))
        else:
            _no_rise(ehvi_grid_batched(mu1, var1, front1, r), ehvi_grid_batched(mu, var, pf, r))


class _Problem:
    def __init__(self, n_obj=2):
        self.n_var, self.n_obj = 2, n_obj
        self.xl, self.xu = np.array([-2.0, -2.0]), np.array([2.0, 2.0])


def _stripes_front(spec):
    y1, y2 = spec.stripes
    return np.column_stack([y1[1:-1], y2[1:-1]])


@pytest.mark.parametrize("ehvi", ["reference", "box"])
def test_multi_closure_front_grows_only_by_non_dominated_rows(ehvi):
    opt = MultiSurrogateOptimiser(_Problem(), [0, 0], [10.0, 10.0], ehvi=ehvi, batch_size=3, semantics="exact")
    pf = np.array([[1.0, 5.0], [2.0, 3.0], [4.0, 1.0]])
    cache = host_prep.cached_samples(2, 3, seed=0)
    spec_for = opt._batch_spec_for(pf, cache)
    same = spec_for(np.empty((0, 2)))
    ref = ob.spec_ehvi_box([10.0, 10.0], pf) if ehvi == "box" else ob.spec_ehvi([10.0, 10.0], pf, cache, "exact")
    np.testing.assert_array_equal(same.stripes, ref.stripes)
    cases = [(np.array([[3.0, 4.0]]), pf),                                   # dominated: no change
             (np.array([[11.0, 0.5]]), pf),                                  # beyond r: no change
             (np.array([[1.5, 2.0]]), np.array([[1.0, 5.0], [1.5, 2.0], [4.0, 1.0]])),   # dominates [2, 3]
             (np.array([[1.5, 2.0], [0.5, 9.0], [3.0, 4.0]]),
              np.array([[1.0, 5.0], [1.5, 2.0], [4.0, 1.0], [0.5, 9.0]]))]
    for Y_bel, want in cases:
        spec = spec_for(Y_bel)
        ref = (ob.spec_ehvi_box([10.0, 10.0], want) if ehvi == "box"
               else ob.spec_ehvi([10.0, 10.0], want, cache, "exact"))
        np.testing.assert_array_equal(spec.stripes, ref.stripes)
        if ehvi == "reference":
            got = _stripes_front(spec)
            assert {tuple(p) for p in got} == {tuple(p) for p in want}
            assert spec.reserved & _cabi.ACQ_FRONT_VALID


def test_multi_closure_decomposition_g_min_is_the_minimum():
    opt = MultiSurrogateOptimiser(_Problem(), [0, 0], [10.0, 10.0], batch_size=2)
    g = ob.scalarisations.Tchebicheff([0, 0], [10.0, 10.0])
    ref_dir = np.array([0.5, 0.5])
    cache = host_prep.cached_samples(2, 3, seed=0)
    spec_for = opt._batch_spec_for(np.array([[1.0, 5.0]]), cache, ref_dir, g, 2.0)
    assert spec_for(np.empty((0, 2))).best == 2.0
    Y = np.array([[3.0, 3.0], [0.2, 0.4]])
    assert spec_for(Y[:1]).best == min(2.0, float(np.ravel(g(Y[0], ref_dir))[0]))
    assert spec_for(Y).best == min(2.0, *[float(np.ravel(g(y, ref_dir))[0]) for y in Y])


def test_mono_closure_incumbent_is_the_minimum():
    spec_for = MonoSurrogateOptimiser._batch_spec_for(0.7)
    assert spec_for(np.empty((0, 1))).best == 0.7
    assert spec_for(np.array([[0.9]])).best == 0.7
    assert spec_for(np.array([[0.9], [0.3], [0.5]])).best == 0.3
    assert spec_for(np.array([[0.9]])).kind == _cabi.ACQ_EI


def test_batch_size_is_validated():
    for bad in (0, -1, 1.5):
        with pytest.raises(ValueError):
            MultiSurrogateOptimiser(_Problem(), batch_size=bad)
        with pytest.raises(ValueError):
            MonoSurrogateOptimiser(_Problem(), batch_size=bad)
    assert MultiSurrogateOptimiser(_Problem()).batch_size == 1
