"""GPU: the acquisition kernels (K4 + K5) in the tails, against the 50-digit reference (tests/acq_mpmath.py).

(a) The FP64 kernel on controlled posteriors keeps the reference's own arithmetic (rtol 1e-12 against oracle/oracle.py)
    and matches mpmath where that arithmetic is well conditioned.
(b) The FP32 kernel of the fast precision mode, on the fast path's own posteriors, steered into each hard regime (EI
    deep in the lower tail, mostly infeasible constrained pools, HV-PoI below the ideal point, dominated 2-D EHVI
    pools, fronts far from the origin).  Every case asserts that it reaches its regime.
(c) The arg-max: +inf, signed zeros, an all -inf pool, index bases above 2^31 / 2^32 and ties across the CTA, chunk
    and pass boundaries."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi  # noqa: E402
from oracle import oracle as O  # noqa: E402
import acq_mpmath as M  # noqa: E402
from test_gpu_parity import make_problem  # noqa: E402

DEV = "cuda:0"
needs_fast = pytest.mark.skipif(not _cabi.fast_path_available(), reason="fast path not built")
TINY = 1e-280          # below this the exact value is not compared (float64 output, subnormal range)


def _acq64(spec, mu, var, index_base=0):
    """FP64 K4 + K5 on given posteriors (m, G)."""
    a, bv, bi = ob.acquire_from_posterior(spec, np.asarray(mu).T, np.asarray(var).T, DEV, index_base=index_base)
    return a.cpu().numpy(), bv, bi


def _fast(models, spec, pool):
    """FP32 K4 on the fast path's posteriors: (acq, mu (m, G), var (m, G), best_value, best_index)."""
    res = ob.score(models, spec, pool, precision="fast", want_posterior=True, want_acq=True)
    return (res.acq.cpu().numpy(), res.mu.cpu().numpy().T, res.var.cpu().numpy().T, res.best_value,
            res.best_index)


def _fast_posterior(models, pool):
    res = ob.score(models, None, pool, precision="fast", want_posterior=True)
    return res.mu.cpu().numpy().T, res.var.cpu().numpy().T


def _gap_ok(v, rtol=1e-3):
    """True when the top value beats the second by more than rtol (relative): the selection is then determined."""
    w = np.sort(np.where(np.isnan(v), -np.inf, v))
    return w[-1] > 0 and w[-1] - w[-2] > rtol * abs(w[-1])


def _check_ei_contract(got, bi, want):
    """rtol 1e-3 where the exact value is >= 1e-280, never negative, the exact arg-max when it is determined."""
    assert np.all(got >= 0), got[got < 0][:5]
    big = want >= TINY
    np.testing.assert_allclose(got[big], want[big], rtol=1e-3, atol=0)
    assert np.all(got[~big] <= 1e-270)
    if _gap_ok(want):
        assert bi == M.argmax_lowest_index(want), (bi, M.argmax_lowest_index(want), got[bi], want.max())


def _best_for_band(mu, s, lo, hi):
    """The `best` that puts the most candidates at g = (best - mu) / s in [lo, hi] (candidates j: best = mu_j + c s_j)."""
    mid = 0.5 * (lo + hi)
    cand = mu + mid * s
    sub = cand[np.linspace(0, len(cand) - 1, min(len(cand), 1500)).astype(int)]
    g = (sub[:, None] - mu[None, :]) / s[None, :]
    count = ((g >= lo) & (g <= hi)).sum(1)
    return float(sub[np.argmax(count)])


# ------------------------------------------------------------------------------------------
# (a) FP64 K4 on controlled posteriors
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("var_eps", [0.0, 1e-6])
def test_fp64_ei_sweep(var_eps):
    g = np.concatenate([np.linspace(-38.0, 38.0, 761), [0.0]])
    var = np.tile([1.0, 0.04, 1e-15, 0.0, 2.5], len(g) // 5 + 1)[:len(g)]
    best = 0.25
    s = np.sqrt(var + var_eps)
    mu = best - g * (s + 1e-10)
    mu[-1] = best                                           # mu exactly at best
    mu = np.concatenate([mu, [np.nan, 0.1, 0.2]])
    var = np.concatenate([var, [0.5, np.nan, 1e-15]])
    got, bv, bi = _acq64(ob.spec_ei(best, var_eps), mu[:, None], var[:, None])
    want = O.expected_improvement(mu, var, best, var_eps)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.isnan(got).sum() == 2
    # beyond |g| = 10, g Phi(g) + phi(g) cancels by ~g^2: the last-ulp differences of CUDA's and scipy's erfc grow past
    # 1e-12 there (5.5e-12 at g = -20), and below g ~ -37 the value is subnormal
    gg = (best - mu) / (np.sqrt(var + var_eps) + 1e-10)
    mid = ~(np.abs(gg) > 10)
    np.testing.assert_allclose(got[mid], want[mid], rtol=1e-12, atol=0, equal_nan=True)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-300, equal_nan=True)
    assert bi == O.argmax_lowest_index(want) and bv == got[bi]
    # well conditioned (|g| <= 5, sigma not at the floor): the exact value
    ok = (np.abs(gg) <= 5) & (var + var_eps > 1e-12)
    assert ok.sum() > 50
    np.testing.assert_allclose(got[ok], M.expected_improvement(mu[ok], var[ok], best, var_eps), rtol=1e-12)


def test_fp64_constrained_pareto_and_hv_poi_edges():
    rng = np.random.default_rng(0)
    m = 400
    mu = np.column_stack([rng.uniform(-1, 1, m), rng.uniform(-3, 3, (m, 2))])
    var = np.column_stack([rng.uniform(0.01, 1, m), rng.uniform(0.01, 1, (m, 2))])
    mu[:20, 1] = 0.0                                        # constraint mean exactly on the boundary
    var[20:40, 0] = 0.0
    var[40:60, 0] = 1e-15
    mu[60:80, 0] = 0.3                                      # at best
    mu[80, 2] = np.nan
    got, _, bi = _acq64(ob.spec_constrained_ei(0.3, 2), mu, var)
    want = O.constrained_ei(mu, var, 0.3)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0, equal_nan=True)
    assert bi == O.argmax_lowest_index(want)
    ok = var[:, 0] > 1e-12
    np.testing.assert_allclose(got[ok], M.constrained_ei(mu[ok], var[ok], 0.3), rtol=1e-12, equal_nan=True)
    got, _, bi = _acq64(ob.spec_pareto_ei(0.3), mu[:, :2][:, ::-1], var[:, :2][:, ::-1])
    want = O.pareto_ei(mu[:, 1], mu[:, 0], var[:, 0], 0.3)
    np.testing.assert_allclose(got, want, rtol=1e-12, equal_nan=True)
    # HV-PoI: means on a cell bound, on a front coordinate, a 1-point front and duplicate coordinates
    for PF in (np.array([[0.4, 0.5]]), np.array([[.1, .9], [.4, .5], [.4, .5], [.8, .5], [.8, .2]])):
        cells = ob.host_prep.decompose_into_cells(PF, [0.0, 0.0], [1.0, 1.0])
        mh = rng.uniform(-0.2, 1.2, (m, 2))
        mh[:10] = PF[0]
        mh[10:20, 0] = 0.0
        mh[20:30] = [1.0, 1.0]
        vh = rng.uniform(0.001, 0.2, (m, 2))
        got, _, bi = _acq64(ob.spec_hv_poi(cells), mh, vh)
        want = O.hv_poi_batched(mh, vh, cells)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-300)
        assert bi == O.argmax_lowest_index(want)
        np.testing.assert_allclose(got, M.hv_poi(mh, vh, cells), rtol=1e-10, atol=1e-14 * want.max())


@pytest.mark.parametrize("semantics", ["reference", "exact"])
def test_fp64_ehvi2d_edges(semantics):
    rng = np.random.default_rng(1)
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    for PF in (np.array([[0.4, 0.5]]), np.array([[.1, .9], [.4, .5], [.4, .5], [.6, .5], [.8, .2]])):
        r = np.array([1.0, 1.0])
        spec = ob.spec_ehvi(r, PF, cache, semantics)
        mu = rng.uniform(0.0, 1.2, (300, 2))
        mu[:10] = PF[-1]
        mu[10:20] = r
        mu[20:30, 1] = PF[0, 1]
        var = rng.uniform(0.002, 0.1, (300, 2))
        got, _, bi = _acq64(spec, mu, var)
        want = O.ehvi_batched(mu[:, 0], mu[:, 1], var[:, 0], var[:, 1], PF, r, cache, semantics)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-15 * np.abs(want).max())
        assert bi == O.argmax_lowest_index(want)
        exact = M.ehvi2d_posterior(spec.stripes, mu, var, semantics, spec.cache_c)
        np.testing.assert_allclose(got, exact, rtol=1e-9, atol=1e-12 * np.abs(exact).max())


# ------------------------------------------------------------------------------------------
# (b) FP32 K4 on the fast path's own posteriors
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gp2():
    """Two f8c models at the C2-like shape and a counter pool of 4096 candidates."""
    X, Y, ells, sf2 = make_problem(256, 10)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    pool = ob.CandidatePool.counter(4096, np.zeros(10), np.ones(10), seed=11)
    mu, var = _fast_posterior(models, pool)
    return X, Y, models, pool, mu, var


@needs_fast
@pytest.mark.parametrize("regime", ["band", "deep"])
def test_fp32_ei_tail(gp2, regime):
    X, Y, models, pool, mu, var = gp2
    s = np.sqrt(var[:, 0])
    if regime == "band":
        best = _best_for_band(mu[:, 0], s, -14.0, -12.0)
    else:
        best = float(np.min(mu[:, 0] - 20.0 * s))              # every candidate at g < -20
    got, mu_f, var_f, bv, bi = _fast(models[:1], ob.spec_ei(best), pool)
    assert np.array_equal(mu_f[:, 0], mu[:, 0]) and np.array_equal(var_f[:, 0], var[:, 0])
    g = (best - mu[:, 0]) / (s + 1e-10)
    if regime == "band":
        assert ((g >= -14) & (g <= -12)).sum() >= 100
    want = M.expected_improvement(mu[:, 0], var[:, 0], best)
    if regime == "deep":
        assert g.max() < -12 and _gap_ok(want)
    _check_ei_contract(got, bi, want)
    f64, _, bi64 = _acq64(ob.spec_ei(best), mu[:, :1], var[:, :1])
    assert bi == bi64 or not _gap_ok(want)


def _near_training(X, m, rng, spread=0.03):
    return np.clip(X[rng.integers(0, len(X), m)] + rng.normal(0, spread, (m, X.shape[1])), 0, 1)


@needs_fast
def test_fp32_ei_offset_best():
    """best ~ 1e3 and improvements best - mu ~ 1e-2: best - mu must be formed before the cast to FP32 (casting mu and
    best first moves it by up to ulp(1e3) / 2 = 3e-5, 3e-3 of the improvement).  The pool sits next to the training
    points, whose targets are 1e3 + 0.05 f(x): every cluster of candidates shares a mean near its point's target."""
    X, Y, ells, sf2 = make_problem(128, 4)
    gp = ob.GPModel(X, 1000.0 + 0.05 * Y[:, 1], 0.5 * np.ones(4), 1e-4, device=DEV)
    pool = ob.CandidatePool.explicit(_near_training(X, 8192, np.random.default_rng(2), 0.005), device=DEV)
    mu, var = _fast_posterior([gp], pool)
    m0 = np.sort(mu[:, 0])
    # best 0.02 above the window of means that holds the most candidates in (best - 0.02, best - 0.002)
    count = np.searchsorted(m0, m0 + 0.018) - np.arange(len(m0))
    best = float(m0[np.argmax(count)] + 0.02)
    imp = best - mu[:, 0]
    assert abs(best) > 900 and ((imp > 0.002) & (imp < 0.02)).sum() >= 20, count.max()
    got, _, _, bv, bi = _fast([gp], ob.spec_ei(best), pool)
    _check_ei_contract(got, bi, M.expected_improvement(mu[:, 0], var[:, 0], best))


@needs_fast
def test_fp32_constrained_ei_all_infeasible(gp2):
    X, Y, models, pool, _, _ = gp2
    rng = np.random.default_rng(3)
    cons = [ob.GPModel(X, Y[:, 1] + 30.0, np.full(10, 0.8), 900.0, device=DEV),
            ob.GPModel(X, Y[:, 0] + 25.0, np.full(10, 0.9), 625.0, device=DEV)]
    first = ob.CandidatePool.explicit(_near_training(X, 8192, rng), device=DEV)
    mu, var = _fast_posterior([models[0]] + cons, first)
    logpof = sum(np.log10(np.maximum(M.probability_of_feasibility(mu[:, c], var[:, c]), 1e-300)) for c in (1, 2))
    keep = np.flatnonzero(logpof < -40)[:2048]
    assert len(keep) >= 500
    pool2 = ob.CandidatePool.explicit(first.X[keep], device=DEV)
    mu, var = _fast_posterior([models[0]] + cons, pool2)
    best = _best_for_band(mu[:, 0], np.sqrt(var[:, 0]), -2.0, 2.0)
    spec = ob.spec_constrained_ei(best, 2)
    got, _, _, bv, bi = _fast([models[0]] + cons, spec, pool2)
    want = M.constrained_ei(mu, var, best)
    pof = M.probability_of_feasibility(mu[:, 1], var[:, 1]) * M.probability_of_feasibility(mu[:, 2], var[:, 2])
    assert np.all(pof < 1e-40) and (want >= TINY).sum() >= 100 and _gap_ok(want)
    _check_ei_contract(got, bi, want)


@needs_fast
def test_fp32_pareto_ei_tail(gp2):
    X, Y, models, pool, mu, var = gp2
    best = float(np.min(mu[:, 1] - 16.0 * np.sqrt(var[:, 1] + 1e-6)))
    got, _, _, bv, bi = _fast(models, ob.spec_pareto_ei(best), pool)
    want = M.pareto_ei(mu[:, 0], mu[:, 1], var[:, 1], best)
    assert (want >= TINY).sum() >= 100 and _gap_ok(want)
    big = np.abs(want) >= TINY
    np.testing.assert_allclose(got[big], want[big], rtol=1e-3)
    assert np.all(np.sign(got[big]) == np.sign(want[big]))
    assert bi == M.argmax_lowest_index(want)


@needs_fast
def test_fp32_hv_poi_below_the_ideal_point(gp2):
    X, Y, models, pool, _, _ = gp2
    rng = np.random.default_rng(4)
    first = ob.CandidatePool.explicit(_near_training(X, 8192, rng, 0.02), device=DEV)
    mu, var = _fast_posterior(models, first)
    sd = np.sqrt(var + 1e-5)
    # the ideal point 6 sigma above the median candidate: keep the candidates 4..8 sigma below it in both objectives
    ideal = np.median(mu + 6.0 * sd, axis=0)
    z = (ideal[None, :] - mu) / sd
    keep = np.flatnonzero(np.all((z >= 4) & (z <= 8), axis=1))[:2048]
    assert len(keep) >= 200
    pool2 = ob.CandidatePool.explicit(first.X[keep], device=DEV)
    span = np.abs(mu).max(0) + 1.0
    PF = ideal + span * np.array([[.1, .9], [.4, .5], [.8, .2]])
    cells = ob.host_prep.decompose_into_cells(PF, ideal, ideal + span)
    got, mu2, var2, bv, bi = _fast(models, ob.spec_hv_poi(cells), pool2)
    want = M.hv_poi(mu2, var2, cells)
    assert np.all(got >= 0)
    big = want >= 1e-6 * want.max()
    assert big.sum() >= 50
    np.testing.assert_allclose(got[big], want[big], rtol=1e-3)
    assert _gap_ok(want) and bi == M.argmax_lowest_index(want)


def _dominating_front(mu, var, margin):
    """The non-dominated points of mu - margin * sigma: every candidate is dominated by the front by >= margin sigma
    in every objective, and the candidates whose own point is on the front sit exactly at that margin."""
    PF = ob.host_prep.calc_pf(mu - margin * np.sqrt(var))
    z = (mu[:, None, :] - PF[None, :, :]) / np.sqrt(var)[:, None, :]
    assert np.all(np.any(np.all(z >= margin * (1 - 1e-12), axis=2), axis=1))
    return PF


def _ehvi_fp32_vs_fp64(models, spec, pool, dominated=False, nonneg=True):
    got, mu, var, bv, bi = _fast(models, spec, pool)
    f64, _, bi64 = _acq64(spec, mu, var)
    scale = np.abs(f64).max()
    assert scale > 0
    np.testing.assert_allclose(got, f64, rtol=0, atol=1e-3 * scale)
    if nonneg and (spec.semantics == "exact" or spec.kind == _cabi.ACQ_EHVI_BOX):
        assert np.all(got >= 0)
    if dominated and _gap_ok(f64):
        assert bi == bi64, (bi, bi64)
    return got, bv, bi


def _check_fused(models, spec, pool, got, bv, bi):
    """The fused f8c epilogue against the unfused K4 launch: bit-identical values and selection."""
    if not all(g.plane_format == "f8c" for g in models):
        return False
    before = _cabi.Context.get(0).launch_count()
    fused = ob.score(models, spec, pool, precision="fast", want_acq=True)
    n_fused = _cabi.Context.get(0).launch_count() - before
    plain = ob.score(models, spec, pool, precision="fast", want_acq=True, want_posterior=True)
    n_plain = _cabi.Context.get(0).launch_count() - before - n_fused
    assert n_fused < n_plain
    a_f = fused.acq.cpu().numpy()
    if spec.semantics == "exact":
        assert np.array_equal(a_f, got)
        assert (fused.best_value, fused.best_index) == (bv, bi)
    else:
        # model 1 runs the mean-only kernel, whose FP32 mean is summed in another order (1e-6 of the scale)
        np.testing.assert_allclose(a_f, got, rtol=1e-4, atol=1e-5 * np.abs(got).max())
        assert fused.best_value == a_f[fused.best_index] == np.nanmax(a_f)
    return True


@needs_fast
@pytest.mark.parametrize("semantics", ["reference", "exact"])
@pytest.mark.parametrize("case", ["natural", "dominated", "offset", "beyond_r", "improper"])
def test_fp32_ehvi2d(gp2, semantics, case):
    X, Y, models, pool, mu, var = gp2
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    if case == "dominated":
        if semantics == "reference":
            pytest.skip("the reference semantics' 'sigma' (var0 * C) has no dominance margin in sigma units")
        PF, r = _dominating_front(mu, var, 8.0), mu.max(0) + 1.0
    elif case == "offset":
        if semantics == "reference":
            pytest.skip("C01 < 0 for this cache: the reference's 'sigma' of objective 1 is negative, every value 0")
        PF, r = PF + 1000.0, r + 1000.0                        # the front 1e3 above the means (unit spread)
    elif case == "beyond_r":
        # a front point with f1 > r0 (a user-given max_point is not clipped to): y1 rises along the stripes
        PF = np.vstack([PF, [r[0] + 0.2, PF[:, 1].min() - 0.1]])
    elif case == "improper":
        # a duplicate point, a dominated point and a duplicate f2: the stripes are not monotone either
        PF = np.vstack([PF, PF[2], PF[3] + [0.05, 0.0], PF[1] + 0.03])
    spec = ob.spec_ehvi(r, PF, cache, semantics)
    proper = case in ("natural", "dominated", "offset")
    if not proper:
        assert np.any(np.diff(spec.stripes[0][:-1]) > 0)        # the regime: y1 is not non-increasing
    got, bv, bi = _ehvi_fp32_vs_fp64(models, spec, pool, dominated=case == "dominated", nonneg=proper)
    assert _check_fused(models, spec, pool, got, bv, bi)


@needs_fast
def test_fp32_box_dominated(gp2):
    X, Y, models, pool, mu, var = gp2
    PF = _dominating_front(mu, var, 8.0)
    _ehvi_fp32_vs_fp64(models, ob.spec_ehvi_box(mu.max(0) + 1.0, PF), pool, dominated=True)


@needs_fast
@pytest.mark.parametrize("case", ["natural", "offset"])
def test_fp32_box_and_crude_3d(case):
    X, Y, ells, sf2 = make_problem(256, 6, k=3)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(3)]
    pool = ob.CandidatePool.counter(4096, np.zeros(6), np.ones(6), seed=13)
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0) + 0.1
    if case == "offset":
        PF, r = PF + 1000.0, r + 1000.0
    _ehvi_fp32_vs_fp64(models, ob.spec_ehvi_box(r, PF), pool)
    cache = ob.host_prep.cached_samples(3, 5, seed=0)
    for sem in ("reference", "exact"):
        _ehvi_fp32_vs_fp64(models, ob.spec_ehvi3d(r, PF, cache, sem), pool)


# ------------------------------------------------------------------------------------------
# (c) K5 selection edges
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base", [0, (1 << 31) + 7, (1 << 32) + 3])
def test_argmax_inf_signed_zero_and_index_base(base):
    m = 3 * 256 + 11
    # Pareto EI = mu_pareto * EI: with EI = 0 (var 0, mu above best) the sign of mu_pareto gives -0.0 or +0.0
    mu = np.column_stack([np.ones(m), np.full(m, 5.0)])
    var = np.column_stack([np.ones(m), np.zeros(m)])
    mu[:, 0] = np.where(np.arange(m) % 3 == 1, 1.0, -1.0)
    mu[:300, 0] = np.nan
    first_zero = 300                                        # index 300: mu_pareto = -1 -> -0.0; 301: +0.0
    got, bv, bi = _acq64(ob.spec_pareto_ei(0.0), mu, var, index_base=base)
    assert np.all(got[first_zero:] == 0) and np.signbit(got[first_zero]) and not np.signbit(got[301])
    assert bi == base + first_zero and bv == 0.0
    # +inf (var = inf) wins over everything, the lowest of two +inf
    var2 = var.copy()
    var2[[500, 700], 1] = np.inf
    got, bv, bi = _acq64(ob.spec_pareto_ei(0.0), np.abs(np.nan_to_num(mu, nan=1.0)), var2, index_base=base)
    assert bv == np.inf and bi == base + 500
    # all -inf: the lowest index, value -inf
    mu3 = np.column_stack([np.full(m, -np.inf), np.zeros(m)])
    got, bv, bi = _acq64(ob.spec_pareto_ei(1.0), mu3, np.ones((m, 2)), index_base=base)
    assert np.all(got == -np.inf) and bv == -np.inf and bi == base


@needs_fast
def test_ties_across_cta_chunk_and_pass_boundaries():
    """Two bit-identical copies of the winner, one in the first 2^20 rows and one past 2^22 (the winner of each precision
    for that precision's pass): the lower one wins, fused and unfused, through the device-pool passes (2^22) and
    propose_host's passes (2^20)."""
    X, Y, ells, sf2 = make_problem(128, 10)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    spec = ob.spec_ehvi(Y.max(0), ob.host_prep.calc_pf(Y), ob.host_prep.cached_samples(2, 5, seed=0), "exact")
    m = (1 << 22) + 4096
    X0 = np.random.default_rng(5).random((m, 10))
    lo, hi = (1 << 20) - 1, (1 << 22) + 77
    for precision in ("fp64", "fast"):
        w = ob.score(models, spec, ob.CandidatePool.explicit(X0, device=DEV), precision=precision).best_index
        Xc = X0.copy()
        Xc[[lo, hi]] = X0[w]
        Xc[w] = X0[w + 1 if w + 1 not in (lo, hi) else w + 2]
        pool = ob.CandidatePool.explicit(Xc, device=DEV)
        res = ob.score(models, spec, pool, precision=precision, want_posterior=True, want_acq=True)
        mu, var, acq = res.mu.cpu().numpy(), res.var.cpu().numpy(), res.acq.cpu().numpy()
        assert np.array_equal(mu[:, lo], mu[:, hi]) and np.array_equal(var[:, lo], var[:, hi])
        assert acq[lo] == acq[hi]
        assert res.best_index == O.argmax_lowest_index(acq) == lo
        fused = ob.score(models, spec, pool, precision=precision, want_acq=True)
        assert (fused.best_index, fused.best_value) == (res.best_index, res.best_value)
        assert np.array_equal(fused.acq.cpu().numpy(), acq)
        hv, hi_idx = ob.propose_host(models, spec, Xc, precision=precision)
        assert (hi_idx, hv) == (res.best_index, res.best_value)
