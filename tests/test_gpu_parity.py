"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs, against the committed golden fixtures minted from the reference's own code, and
through size-independent properties.  Tolerances: FP64 mode rtol 1e-6 (north_star) with the
atol the SURVEY derives (section 7, "variance cancellation"): atol = 1e-7 * sigma_f on sigma."""
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
from oracle import oracle as O  # noqa: E402

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def zdt1(X):
    f1 = X[:, 0]
    g = 1 + 9.0 / (X.shape[1] - 1) * X[:, 1:].sum(1)
    return np.column_stack([f1, g * (1 - np.sqrt(f1 / g))])


def make_problem(n, d, seed=0, k=2):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    if k == 2:
        Y = zdt1(X) if d > 1 else np.column_stack([X[:, 0], 1 - X[:, 0] ** 2])
    else:
        Y = np.column_stack([np.cos(X[:, :2].sum(1)) + 1.5, np.sin(X[:, 1:3].sum(1)) + 1.5, X[:, -1] + X[:, 0] ** 2])
    ells = [(0.7 + 0.1 * i) * np.ones(d) * (1 + 0.05 * np.arange(d)) for i in range(k)]
    sf2 = [1.0 + i for i in range(k)]
    return X, Y, ells, sf2


# ------------------------------------------------------------------------------------------
# candidate generator
# ------------------------------------------------------------------------------------------
def test_counter_pool_bit_exact():
    lo, hi = np.array([-2.0, 0.0, 1.0]), np.array([2.0, 5.0, 1.5])
    pool = ob.CandidatePool.counter(5000, lo, hi, seed=7, index_base=123456789012)
    got = pool.rows(123456789012, 5000, DEV).cpu().numpy()
    want = O.candidates_from_counter(7, 123456789012, 5000, lo, hi)
    assert np.array_equal(got, want)
    sh = pool.shard(1, 4)
    assert sh.index_base == 123456789012 + 1250 and sh.m == 1250
    assert np.array_equal(sh.rows(sh.index_base, 10, DEV).cpu().numpy(), want[1250:1260])


# ------------------------------------------------------------------------------------------
# K3: refresh
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(1, 1), (20, 2), (100, 2), (128, 3), (129, 5), (256, 10), (700, 12)])
def test_refresh_vs_oracle(n, d):
    X, Y, ells, sf2 = make_problem(n, d)
    gp = ob.GPModel(X, Y[:, 1], ells[1], sf2[1], device=DEV)
    st = O.gp_fit_state(X, Y[:, 1], ells[1], sf2[1], form="direct")
    L = gp.L.cpu().numpy()
    np.testing.assert_allclose(L, st["L"], rtol=1e-7, atol=1e-9)
    Linv = gp.Linv.cpu().numpy()
    assert np.allclose(np.triu(Linv, 1), 0)
    np.testing.assert_allclose(Linv @ st["L"], np.eye(n), atol=1e-6)
    # alpha: compare through K alpha = y (alpha itself is ill-conditioned)
    K = st["L"] @ st["L"].T
    np.testing.assert_allclose(K @ gp.alpha.cpu().numpy(), Y[:, 1], rtol=1e-6, atol=1e-6)


def test_refresh_not_pd_raises_and_retries():
    X = np.array([[0.1, 0.2], [0.1, 0.2], [0.5, 0.5]])   # duplicate rows, jitter 0 -> singular
    y = np.array([1.0, 1.0, 2.0])
    gp = ob.GPModel(X, y, [1.0, 1.0], 1.0, jitter=0.0, device=DEV, refresh=False, max_jitter_tries=0)
    with pytest.raises(_cabi.NotPositiveDefinite):
        gp.refresh()
    gp2 = ob.GPModel(X, y, [1.0, 1.0], 1.0, jitter=0.0, device=DEV)     # jitchol-style retry
    assert gp2.effective_jitter > 0
    mu, var = gp2.predict(X)
    np.testing.assert_allclose(mu[:, 0], y, atol=1e-3)


# ------------------------------------------------------------------------------------------
# K1 + K2: posterior, FP64 mode
# ------------------------------------------------------------------------------------------
POSTERIOR_CASES = [
    # (n, d, m, kernel)       config it mirrors
    (20, 2, 1000, "matern52"),     # C1 README first iteration
    (119, 2, 4096, "matern52"),    # C1 last iteration (ill-conditioned)
    (100, 2, 5000, "matern52"),    # C3 BNH, N_max = 100
    (256, 10, 1 << 14, "matern52"),  # C2
    (512, 12, 1 << 13, "matern52"),  # C4
    (1024, 10, 1 << 12, "matern52"),  # C5
    (300, 7, 3000, "rbf"),
    (1, 3, 100, "matern52"),
]


@pytest.mark.parametrize("n,d,m,kernel", POSTERIOR_CASES)
def test_posterior_fp64_vs_oracle(n, d, m, kernel):
    X, Y, ells, sf2 = make_problem(n, d)
    kid = O.KERNEL_MATERN52 if kernel == "matern52" else O.KERNEL_RBF
    rng = np.random.default_rng(5)
    Xc = rng.random((m, d)) * 1.2 - 0.1
    Xc[: min(n, 8)] = X[: min(n, 8)]             # candidates ON training points: sigma -> floor
    for i in range(2):
        gp = ob.GPModel(X, Y[:, i], ells[i], sf2[i], kernel=kernel, device=DEV)
        st = O.gp_fit_state(X, Y[:, i], ells[i], sf2[i], kernel=kid)
        mu_o, var_o = O.gp_posterior(st, Xc)
        mu, var = ob.posterior([gp], Xc)
        mu, var = mu[0].cpu().numpy(), var[0].cpu().numpy()
        scale = max(1.0, np.abs(mu_o).max())
        np.testing.assert_allclose(mu, mu_o, rtol=1e-6, atol=1e-7 * scale)
        np.testing.assert_allclose(np.sqrt(var), np.sqrt(var_o), rtol=1e-6, atol=2e-6 * np.sqrt(sf2[i]))
        assert var.min() >= 1e-15
        # both model surfaces
        m1, v1 = gp.predict(Xc[:50])
        assert m1.shape == (50, 1) and v1.shape == (50, 1)
        np.testing.assert_allclose(m1[:, 0], mu[:50], rtol=0, atol=0)
        m2, s2 = gp.predict(Xc[:50], return_std=True)
        assert m2.shape == (50,) and s2.shape == (50,)
        np.testing.assert_allclose(s2[8:], np.sqrt(v1[8:, 0]), rtol=1e-12)


def test_posterior_f32_candidates_and_generated_pool():
    n, d, m = 200, 6, 3000
    X, Y, ells, sf2 = make_problem(n, d)
    gp = ob.GPModel(X, Y[:, 0], ells[0], sf2[0], device=DEV)
    st = O.gp_fit_state(X, Y[:, 0], ells[0], sf2[0])
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=3, index_base=10 ** 9)
    mu, var = ob.posterior([gp], pool)
    Xc = O.candidates_from_counter(3, 10 ** 9, m, np.zeros(d), np.ones(d))
    mu_o, var_o = O.gp_posterior(st, Xc)
    np.testing.assert_allclose(mu[0].cpu().numpy(), mu_o, rtol=1e-6, atol=1e-7)
    X32 = torch.as_tensor(Xc.astype(np.float32)).to(DEV)
    mu32, _ = ob.posterior([gp], ob.CandidatePool.explicit(X32))
    mu_o32, _ = O.gp_posterior(st, Xc.astype(np.float32).astype(np.float64))
    np.testing.assert_allclose(mu32[0].cpu().numpy(), mu_o32, rtol=1e-6, atol=1e-7)


def test_posterior_interpolates_training_set():
    """Size-independent property: a noise-free GP reproduces y at X with sigma at the floor."""
    n, d = 384, 8
    X, Y, ells, sf2 = make_problem(n, d)
    gp = ob.GPModel(X, Y[:, 1], ells[1], sf2[1], device=DEV)
    mu, var = gp.predict(X)
    np.testing.assert_allclose(mu[:, 0], Y[:, 1], atol=5e-5)
    assert var.max() < 1e-5 and var.min() >= 1e-15


# ------------------------------------------------------------------------------------------
# K4: acquisition arithmetic against the reference-minted fixtures
# ------------------------------------------------------------------------------------------
def _close(got, want, rtol=1e-6, atol_scale=1e-9):
    want = np.asarray(want)
    ok = np.isfinite(want)
    np.testing.assert_allclose(np.asarray(got)[ok], want[ok], rtol=rtol, atol=atol_scale * max(1e-300, np.abs(want[ok]).max()))


def test_ehvi_reference_golden(golden):
    mu, var = golden["acq_in_mu2"], golden["acq_in_var2"]
    spec = ob.spec_ehvi(golden["acq_in_ref"], golden["acq_out_calc_pf"], golden["acq_in_cache2"])
    acq, bv, bi = ob.acquire_from_posterior(spec, mu.T, var.T, DEV)
    want = golden["acq_out_EHVI"]
    _close(acq.cpu().numpy(), want, rtol=1e-6, atol_scale=1e-8)
    finite = np.where(np.isnan(want), -np.inf, want)
    assert bi == int(np.argmax(finite))


def test_ehvi_exact_semantics(golden):
    mu, var = golden["acq_in_mu2"], golden["acq_in_var2"]
    PF, r = golden["acq_out_calc_pf"], golden["acq_in_ref"]
    spec = ob.spec_ehvi(r, PF, golden["acq_in_cache2"], semantics="exact")
    acq, _, _ = ob.acquire_from_posterior(spec, mu.T, var.T, DEV)
    want = O.ehvi2d_aux_batched(PF, r, mu[:, 0], mu[:, 1], np.sqrt(var[:, 0]), np.sqrt(var[:, 1]), exact=True)
    _close(acq.cpu().numpy(), want, rtol=1e-6, atol_scale=1e-10)
    # minus the extra stripe it is the reference's EHVI_2D_aux with true stds
    assert np.all(acq.cpu().numpy() >= golden["acq_out_EHVI_2D_aux_truestd"] - 1e-9)
    # anchor (SURVEY 8c): textbook value
    specA = ob.spec_ehvi([1, 1], np.array([[.1, .9], [.4, .5], [.8, .2]]), golden["acq_in_cache2"], "exact")
    a, _, _ = ob.acquire_from_posterior(specA, [[.3], [.6]], [[.04], [.09]], DEV)
    np.testing.assert_allclose(a.cpu().numpy(), [0.0768782210398855], rtol=1e-10)


@pytest.mark.parametrize("name", O.SCALARISATIONS)
def test_expected_decomposition_golden(golden, name):
    from optimobo_b200 import scalarisations as S
    mu, var = golden["acq_in_mu2"], golden["acq_in_var2"]
    kw = dict(p=8) if name == "ExponentialWeightedCriterion" else {}
    obj = getattr(S, name)(golden["ed_in_ideal"], golden["ed_in_max"], **kw)
    for key, cache in (("ed_out_", golden["acq_in_cache2"]), ("ed8_out_", golden["ed_in_cache8"])):
        spec = ob.spec_expected_decomposition(golden["ed_in_w"], obj, golden[f"ed_in_gmin_{name}"][0], cache)
        acq, _, _ = ob.acquire_from_posterior(spec, mu.T, var.T, DEV)
        _close(acq.cpu().numpy(), golden[key + name], rtol=1e-6, atol_scale=1e-12)


def test_ehvi3d_golden(golden):
    spec = ob.spec_ehvi3d(golden["e3_in_ref"], golden["e3_in_pf"], golden["e3_in_cache"])
    np.testing.assert_allclose(spec.best, golden["e3_in_sminus"][0], rtol=1e-12)
    acq, _, _ = ob.acquire_from_posterior(spec, golden["e3_in_mu"].T, golden["e3_in_var"].T, DEV)
    _close(acq.cpu().numpy(), golden["e3_out_EHVI_3D"], rtol=1e-9)


def test_ei_family_golden(golden):
    mu, var = golden["acq_in_mu2"], golden["acq_in_var2"]
    best = golden["ei_in_best"][0]
    a, _, _ = ob.acquire_from_posterior(ob.spec_ei(best, 0.0), mu[:, :1].T, var[:, :1].T, DEV)
    _close(a.cpu().numpy(), golden["ei_out_mono"], rtol=1e-9, atol_scale=1e-14)
    a, _, _ = ob.acquire_from_posterior(ob.spec_ei(best, 1e-6), mu[:, :1].T, var[:, :1].T, DEV)
    _close(a.cpu().numpy(), golden["ei_out_parego"], rtol=1e-9)
    _close(a.cpu().numpy(), golden["ei_out_keep"], rtol=1e-9)
    # KEEP: models = [pareto, scalar] = golden columns [1, 0]
    a, _, _ = ob.acquire_from_posterior(ob.spec_pareto_ei(best), mu[:, [1, 0]].T, var[:, [1, 0]].T, DEV)
    _close(a.cpu().numpy(), golden["pei_out_keep"], rtol=1e-9)
    a, _, _ = ob.acquire_from_posterior(ob.spec_constrained_ei(best, 2), golden["cei_in_mu"].T, golden["cei_in_var"].T, DEV)
    _close(a.cpu().numpy(), golden["cei_out_c2"], rtol=1e-9, atol_scale=1e-14)


def test_hv_poi_golden(golden):
    cells = ob.host_prep.decompose_into_cells(golden["acq_out_calc_pf"], golden["emo_in_ideal"], golden["emo_in_max"])
    assert np.array_equal(cells, golden["emo_out_cells"])
    a, _, _ = ob.acquire_from_posterior(ob.spec_hv_poi(cells), golden["acq_in_mu2"].T, golden["acq_in_var2"].T, DEV)
    _close(a.cpu().numpy(), golden["emo_out_poi"], rtol=1e-9, atol_scale=1e-14)


# ------------------------------------------------------------------------------------------
# K5: arg-max semantics
# ------------------------------------------------------------------------------------------
def test_argmax_ties_nan_and_index_base():
    m = 70001
    mu = np.zeros((1, m)); var = np.full((1, m), 0.04)
    mu[0, [5, 40000, 69999]] = -3.0                       # three equal maxima of EI
    _, bv, bi = ob.acquire_from_posterior(ob.spec_ei(0.0), mu, var, DEV, index_base=1000)
    assert bi == 1005
    var[0, 5] = np.nan                                    # NaN is never selected
    _, bv, bi = ob.acquire_from_posterior(ob.spec_ei(0.0), mu, var, DEV, index_base=1000)
    assert bi == 41000 and np.isfinite(bv)
    var[:] = np.nan                                       # all NaN: lowest index, value -inf
    _, bv, bi = ob.acquire_from_posterior(ob.spec_ei(0.0), mu, var, DEV, index_base=1000)
    assert bi == 1000 and bv == -np.inf


# ------------------------------------------------------------------------------------------
# whole path: GP -> acquisition -> arg-max, per config shape
# ------------------------------------------------------------------------------------------
def _oracle_post(X, Y, ells, sf2, Xc, k):
    post = [O.gp_posterior(O.gp_fit_state(X, Y[:, i], ells[i], sf2[i]), Xc) for i in range(k)]
    return np.array([p[0] for p in post]), np.array([p[1] for p in post])


def _check_selection(acq_gpu, acq_oracle, best_index, rtol=1e-6):
    """identical selected candidate whenever the top-two gap exceeds the tolerance (north_star)."""
    a = np.where(np.isnan(acq_oracle), -np.inf, acq_oracle)
    order = np.argsort(-a, kind="stable")
    top, second = a[order[0]], a[order[1]]
    if top - second > rtol * max(abs(top), 1e-300) * 10:
        assert best_index == order[0]
    else:
        assert acq_gpu[best_index] >= np.nanmax(acq_gpu) * (1 - 1e-12) or np.nanmax(acq_gpu) <= 0


@pytest.mark.parametrize("n,d,m", [(256, 10, 1 << 14), (1024, 10, 1 << 12)])
def test_full_path_ehvi(n, d, m):
    X, Y, ells, sf2 = make_problem(n, d)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    lo, hi = np.zeros(d), np.ones(d)
    pool = ob.CandidatePool.counter(m, lo, hi, seed=1)
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    for sem in ("reference", "exact"):
        res = ob.score(models, ob.spec_ehvi(r, PF, cache, sem), pool, want_acq=True)
        Xc = O.candidates_from_counter(1, 0, m, lo, hi)
        mu_o, var_o = _oracle_post(X, Y, ells, sf2, Xc, 2)
        want = O.ehvi_batched(mu_o[0], mu_o[1], var_o[0], var_o[1], PF, r, cache, sem)
        got = res.acq.cpu().numpy()
        np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-7 * np.abs(want).max())
        _check_selection(got, want, res.best_index)
        x, neg, idx = ob.propose(models, ob.spec_ehvi(r, PF, cache, sem), pool)
        assert idx == res.best_index and np.array_equal(x, Xc[idx]) and neg == -res.best_value


def test_full_path_constrained_ei_bnh():
    """C3: BNH, ParEGO_C2 -- agg GP + 2 constraint GPs sharing the inputs, n = 100, d = 2."""
    rng = np.random.default_rng(3)
    n, m = 100, 1 << 15
    lo, hi = np.zeros(2), np.array([5.0, 3.0])
    X = lo + (hi - lo) * rng.random((n, 2))
    f1 = 4 * X[:, 0] ** 2 + 4 * X[:, 1] ** 2
    f2 = (X[:, 0] - 5) ** 2 + (X[:, 1] - 5) ** 2
    g1 = (1 / 25) * ((X[:, 0] - 5) ** 2 + X[:, 1] ** 2 - 25)
    g2 = -1 / 7.7 * ((X[:, 0] - 8) ** 2 + (X[:, 1] + 3) ** 2 - 7.7)
    agg = np.maximum(0.5 * f1 / 150, 0.5 * f2 / 60)
    Ys = np.column_stack([agg, g1, g2])
    ells = [np.array([1.5, 1.0])] * 3
    sf2 = [1.0, 1.0, 1.0]
    models = [ob.GPModel(X, Ys[:, i], ells[i], sf2[i], device=DEV) for i in range(3)]
    pool = ob.CandidatePool.counter(m, lo, hi, seed=11)
    best = agg.min()
    res = ob.score(models, ob.spec_constrained_ei(best, 2), pool, want_acq=True)
    Xc = O.candidates_from_counter(11, 0, m, lo, hi)
    mu_o, var_o = _oracle_post(X, Ys, ells, sf2, Xc, 3)
    want = O.constrained_ei(mu_o.T, var_o.T, best)
    got = res.acq.cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-9 * np.abs(want).max())
    _check_selection(got, want, res.best_index)


def test_full_path_ehvi3d_and_decomposition():
    """C4-shaped: 3 objectives, d = 12."""
    n, d, m = 512, 12, 1 << 12
    X, Y, ells, sf2 = make_problem(n, d, k=3)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(3)]
    lo, hi = np.zeros(d), np.ones(d)
    pool = ob.CandidatePool.counter(m, lo, hi, seed=2)
    Xc = O.candidates_from_counter(2, 0, m, lo, hi)
    mu_o, var_o = _oracle_post(X, Y, ells, sf2, Xc, 3)
    cache = ob.host_prep.cached_samples(3, 5, seed=4)
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0) + 0.5
    res = ob.score(models, ob.spec_ehvi3d(r, PF, cache), pool, want_acq=True)
    want = O.ehvi3d_batched(mu_o.T, var_o.T, r, O.hypervolume(PF, r), cache)
    np.testing.assert_allclose(res.acq.cpu().numpy(), want, rtol=1e-5, atol=1e-8 * np.abs(want).max())
    from optimobo_b200 import scalarisations as S
    ideal, maxp = Y.min(0), Y.max(0)
    w = np.array([0.2, 0.5, 0.3])
    for name in ("Tchebicheff", "PBI", "APD", "WeightedNorm"):
        obj = getattr(S, name)(ideal, maxp)
        gmin = min(obj(y, w)[0] for y in Y)
        res = ob.score(models, ob.spec_expected_decomposition(w, obj, gmin, cache), pool, want_acq=True)
        want = O.expected_decomposition_batched(mu_o.T, var_o.T, w, name, ideal, maxp, gmin, cache)
        np.testing.assert_allclose(res.acq.cpu().numpy(), want, rtol=1e-5, atol=1e-8 * max(np.abs(want).max(), 1e-30))


def test_host_entry_matches_device_entry():
    n, d, m = 128, 4, (1 << 20) + 777          # > one chunk: exercises the double-buffered copies
    X, Y, ells, sf2 = make_problem(n, d)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    spec = ob.spec_ehvi(Y.max(0), ob.host_prep.calc_pf(Y), cache)
    Xh = torch.rand((m, d), dtype=torch.float64, generator=torch.Generator().manual_seed(0)).pin_memory()
    bv, bi = ob.propose_host(models, spec, Xh)
    res = ob.score(models, spec, ob.CandidatePool.explicit(Xh.to(DEV)))
    assert (bv, bi) == (res.best_value, res.best_index)
    bv32, bi32 = ob.propose_host(models, spec, Xh.float().pin_memory())
    assert abs(bv32 - bv) <= 1e-3 * abs(bv) + 1e-12


def test_empty_and_ragged_pools():
    n, d = 50, 3
    X, Y, ells, sf2 = make_problem(n, d)
    gp = ob.GPModel(X, Y[:, 0], ells[0], sf2[0], device=DEV)
    st = O.gp_fit_state(X, Y[:, 0], ells[0], sf2[0])
    for m in (1, 63, 64, 65, 257):
        Xc = np.random.default_rng(m).random((m, d))
        mu, var = ob.posterior([gp], Xc)
        mu_o, var_o = O.gp_posterior(st, Xc)
        np.testing.assert_allclose(mu[0].cpu().numpy(), mu_o, rtol=1e-6, atol=1e-8)
    res = ob.score([gp], ob.spec_ei(0.0), ob.CandidatePool.counter(0, np.zeros(d), np.ones(d)))
    assert res.best_index == -1 and res.best_value == -np.inf


def test_errors_are_loud():
    n, d = 30, 3
    X, Y, ells, sf2 = make_problem(n, d)
    gp = ob.GPModel(X, Y[:, 0], ells[0], sf2[0], device=DEV)
    with pytest.raises(_cabi.OmboError):
        ob.score([gp], ob.spec_ei(0.0), ob.CandidatePool.counter(10, np.zeros(d + 1), np.ones(d + 1)))
    with pytest.raises(ValueError):
        ob.score([gp], ob.spec_pareto_ei(0.0), ob.CandidatePool.counter(10, np.zeros(d), np.ones(d)))

    class Custom(ob.scalarisations.Scalarisation):
        pass
    with pytest.raises(TypeError):
        ob.spec_expected_decomposition([.5, .5], Custom([0, 0], [1, 1]), 0.1, np.zeros((8, 2)))


# ------------------------------------------------------------------------------------------
# fast mode: 16-bit x3 split on tcgen05 (bf16 planes, fp16 for ill-conditioned GPs) (rtol 1e-3, north_star; atol 1e-3 of the output scale
# because sigma -> 0 / mu -> 0 make a pure relative bound meaningless, SURVEY section 7)
# ------------------------------------------------------------------------------------------
FAST_CASES = [(128, 10, 1000), (256, 10, 1 << 14), (512, 12, 1 << 13), (1024, 10, 1 << 13), (700, 7, 5001),
              (100, 4, 129), (1536, 10, 2048)]


@pytest.mark.parametrize("n,d,m", FAST_CASES)
def test_posterior_fast_vs_oracle(n, d, m):
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    X, Y, ells, sf2 = make_problem(n, d)
    Xc = np.random.default_rng(9).random((m, d))
    for i in range(2):
        gp = ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV)
        st = O.gp_fit_state(X, Y[:, i], ells[i], sf2[i])
        mu_o, var_o = O.gp_posterior(st, Xc)
        mu, var = ob.posterior([gp], Xc, precision="fast")
        mu, var = mu[0].cpu().numpy(), var[0].cpu().numpy()
        np.testing.assert_allclose(mu, mu_o, rtol=1e-3, atol=1e-3 * np.abs(mu_o).max())
        np.testing.assert_allclose(np.sqrt(var), np.sqrt(var_o), rtol=1e-3, atol=1e-3 * np.sqrt(sf2[i]))
        # and against the FP64 CUDA path: same tolerance
        mu64, var64 = ob.posterior([gp], Xc, precision="fp64")
        np.testing.assert_allclose(np.sqrt(var), np.sqrt(var64[0].cpu().numpy()), rtol=1e-3, atol=1e-3 * np.sqrt(sf2[i]))
        # bit-reproducible run to run
        mu_b, var_b = ob.posterior([gp], Xc, precision="fast")
        assert torch.equal(mu_b[0].cpu(), torch.as_tensor(mu)) and torch.equal(var_b[0].cpu(), torch.as_tensor(var))


def _in_fresh_process(call, **env):
    """Runs `call` (source text calling a function of this module) in a new interpreter with `env` added to the
    environment: the library reads its knobs once per process, when it creates the device context."""
    code = f"import sys\nsys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\nimport test_gpu_parity as T\nT.{call}\n"
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]


def _posterior_16bit_vs_oracle(n, d, m):
    X, Y, ells, sf2 = make_problem(n, d)
    gp = ob.GPModel(X, Y[:, 0], ells[0], sf2[0], device=DEV)
    assert gp.plane_format in ("bf16x3", "fp16x3"), gp.plane_format      # k_posterior_fast, not the f8c kernel
    st = O.gp_fit_state(X, Y[:, 0], ells[0], sf2[0])
    Xc = np.random.default_rng(n + d).random((m, d))
    sel = np.random.default_rng(1).integers(0, m, min(m, 3000))
    mu_o, var_o = O.gp_posterior(st, Xc[sel])
    mu, var = ob.posterior([gp], Xc, precision="fast")
    mu, var = mu[0].cpu().numpy(), var[0].cpu().numpy()
    np.testing.assert_allclose(mu[sel], mu_o, rtol=1e-3, atol=1e-3 * np.abs(mu_o).max())
    np.testing.assert_allclose(np.sqrt(var[sel]), np.sqrt(var_o), rtol=1e-3, atol=1e-3 * np.sqrt(sf2[0]))
    mu_b, var_b = ob.posterior([gp], Xc, precision="fast")
    assert torch.equal(mu_b[0].cpu(), torch.as_tensor(mu)) and torch.equal(var_b[0].cpu(), torch.as_tensor(var))


@pytest.mark.parametrize("n,d,m", [(100, 4, 129), (512, 12, 3000), (1024, 10, 148 * 128 * 2 + 77), (1536, 7, 2048)])
def test_posterior_fast_16bit_kernel(n, d, m):
    """The 16-bit x3 kernel on the shapes the f8c kernel would otherwise take (OMBO_NO_F8C, in a fresh process):
    ragged m, one to three TMEM passes, n_pad = 128 (two K-blocks: shorter than the operand ring)."""
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    _in_fresh_process(f"_posterior_16bit_vs_oracle({n}, {d}, {m})", OMBO_NO_F8C="1")


def _mean_only_matches_variance_launch(d, ell_bf16, ell_fp16):
    X = np.random.default_rng(d).random((300, d))
    Y = zdt1(X)
    spec = ob.spec_ehvi(Y.max(0), ob.host_prep.calc_pf(Y), ob.host_prep.cached_samples(2, 5, seed=0), "reference")
    pool = ob.CandidatePool.counter(5000, np.zeros(d), np.ones(d), seed=d)
    for ell, fmt in ((ell_bf16, "bf16x3"), (ell_fp16, "fp16x3")):
        models = [ob.GPModel(X, Y[:, i], ell * np.ones(d), 1.0 + i, device=DEV) for i in range(2)]
        assert models[1].plane_format == fmt, (models[1].plane_format, models[1].conditioning)
        # reference semantics never reads model 1's variance: without the posterior requested, model 1 runs the
        # mean-only kernel; with it, k_posterior_fast computes its mean next to the variance
        mean_only = ob.score(models, spec, pool, precision="fast", want_acq=True)
        both = ob.score(models, spec, pool, precision="fast", want_acq=True, want_posterior=True)
        assert torch.equal(mean_only.acq, both.acq)


@pytest.mark.parametrize("d,ell_bf16,ell_fp16", [(6, 0.5, 1.0), (13, 1.0, 3.0), (16, 1.0, 3.0), (24, 1.0, 6.0)])
def test_fast_mean_only_launch_is_bit_identical(d, ell_bf16, ell_fp16):
    """Mean-only launches (k_posterior_mean_fast) give the mean of a variance launch bit for bit, on bf16 and fp16
    planes, with 4 (d <= 12) and 2 (d > 12) candidate rows per generator lane."""
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    _in_fresh_process(f"_mean_only_matches_variance_launch({d}, {ell_bf16}, {ell_fp16})", OMBO_NO_F8C="1")


def test_fast_mode_d16_and_reference_semantics():
    """d > 12 (bf16 x3 planes, 2 rows per generator lane) against the oracle, and the reference-semantics EHVI in fast
    mode (model 1 mean-only) against FP64."""
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    X, Y, ells, sf2 = make_problem(300, 16)
    gp = ob.GPModel(X, Y[:, 0], ells[0] * 2.0, sf2[0], device=DEV)
    st = O.gp_fit_state(X, Y[:, 0], ells[0] * 2.0, sf2[0])
    Xc = np.random.default_rng(3).random((1000, 16))
    mu_o, var_o = O.gp_posterior(st, Xc)
    mu, var = ob.posterior([gp], Xc, precision="fast")
    np.testing.assert_allclose(np.sqrt(var[0].cpu().numpy()), np.sqrt(var_o), rtol=2e-3, atol=2e-3 * np.sqrt(sf2[0]))
    X, Y, ells, sf2 = make_problem(640, 6)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    spec = ob.spec_ehvi(Y.max(0), ob.host_prep.calc_pf(Y), ob.host_prep.cached_samples(2, 5, seed=0), "reference")
    pool = ob.CandidatePool.counter(5000, np.zeros(6), np.ones(6), seed=4)
    fast = ob.score(models, spec, pool, precision="fast", want_acq=True)
    ref = ob.score(models, spec, pool, precision="fp64", want_acq=True)
    a_f, a_r = fast.acq.cpu().numpy(), ref.acq.cpu().numpy()
    np.testing.assert_allclose(a_f, a_r, rtol=5e-3, atol=2e-3 * np.abs(a_r).max())


def test_posterior_fast_rbf_and_high_dim():
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    for n, d, kernel in ((300, 7, "rbf"), (400, 16, "matern52"), (260, 21, "matern52"), (200, 3, "rbf")):
        X, Y, ells, sf2 = make_problem(n, d)
        ell = ells[0] * (2.0 if d > 12 else 1.0)
        # the RBF Gram matrix is numerically singular without noise (cond > 1e12): that regime belongs to
        # the FP64 mode; with a 1e-3 noise term it is a fair fast-mode case
        noise = 1e-3 if kernel == "rbf" else 0.0
        gp = ob.GPModel(X, Y[:, 0], ell, sf2[0], noise=noise, kernel=kernel, device=DEV)
        st = O.gp_fit_state(X, Y[:, 0], ell, sf2[0], sigma_n2=noise,
                            kernel=O.KERNEL_RBF if kernel == "rbf" else O.KERNEL_MATERN52)
        Xc = np.random.default_rng(d).random((2000, d))
        mu_o, var_o = O.gp_posterior(st, Xc)
        mu, var = ob.posterior([gp], Xc, precision="fast")
        np.testing.assert_allclose(mu[0].cpu().numpy(), mu_o, rtol=1e-3, atol=2e-3 * np.abs(mu_o).max())
        np.testing.assert_allclose(np.sqrt(var[0].cpu().numpy()), np.sqrt(var_o), rtol=2e-3, atol=2e-3 * np.sqrt(sf2[0]))
    gp = ob.GPModel(np.random.default_rng(0).random((50, 30)), np.zeros(50), np.ones(30), 1.0, device=DEV)
    with pytest.raises(_cabi.OmboError, match="d <= 24"):
        ob.posterior([gp], np.zeros((4, 30)), precision="fast")


def test_full_path_fast_ehvi_selection():
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    n, d, m = 1024, 10, 1 << 15
    X, Y, ells, sf2 = make_problem(n, d)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    lo, hi = np.zeros(d), np.ones(d)
    pool = ob.CandidatePool.counter(m, lo, hi, seed=1)
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    spec = ob.spec_ehvi(r, PF, cache, "exact")
    fast = ob.score(models, spec, pool, precision="fast", want_acq=True)
    ref = ob.score(models, spec, pool, precision="fp64", want_acq=True)
    a_f, a_r = fast.acq.cpu().numpy(), ref.acq.cpu().numpy()
    np.testing.assert_allclose(a_f, a_r, rtol=5e-3, atol=2e-3 * np.abs(a_r).max())
    # identical selection whenever the top-two gap exceeds the tolerance
    order = np.argsort(-a_r)
    if a_r[order[0]] - a_r[order[1]] > 5e-3 * a_r[order[0]]:
        assert fast.best_index == ref.best_index
    assert a_r[fast.best_index] >= a_r[order[0]] * (1 - 5e-3)


@pytest.mark.parametrize("n,d,m", [(128, 10, 63), (512, 12, 3000), (1024, 10, 148 * 128 + 5), (1024, 10, (1 << 20) + 3)])
def test_fused_acquisition_epilogue_matches_k4(n, d, m):
    """K4 + K5 fused behind the last model's K2 (f8c kernel, 2-D EHVI, no posterior asked for) against the unfused
    launch sequence, which runs when the posterior is also requested: the same FP32 EHVI function on the same mean
    and variance, so values and selection must be identical (util_functions.py:136-167 end to end)."""
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    X, Y, ells, sf2 = make_problem(n, d)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    assert [g.plane_format for g in models] == ["f8c", "f8c"]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    spec = ob.spec_ehvi(r, PF, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
    for pool in (ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=3),
                 ob.CandidatePool.explicit(np.random.default_rng(1).random((min(m, 20000), d)), device=DEV)):
        before = _cabi.Context.get(0).launch_count()
        fused = ob.score(models, spec, pool, precision="fast", want_acq=True)
        n_fused = _cabi.Context.get(0).launch_count() - before
        plain = ob.score(models, spec, pool, precision="fast", want_acq=True, want_posterior=True)
        n_plain = _cabi.Context.get(0).launch_count() - before - n_fused
        only = ob.score(models, spec, pool, precision="fast")
        assert n_fused < n_plain                       # k_acquire did not run
        np.testing.assert_array_equal(fused.acq.cpu().numpy(), plain.acq.cpu().numpy())
        assert (fused.best_index, fused.best_value) == (plain.best_index, plain.best_value) == (only.best_index, only.best_value)
        ref = ob.score(models, spec, pool, precision="fp64", want_acq=True)
        a_r = ref.acq.cpu().numpy()
        np.testing.assert_allclose(fused.acq.cpu().numpy(), a_r, rtol=5e-3, atol=2e-3 * np.abs(a_r).max())


@pytest.mark.parametrize("n,d,m", [(256, 10, 5001), (1024, 10, 148 * 128 + 5)])
def test_fused_acquisition_epilogue_reference_semantics(n, d, m):
    """The reference's default EHVI (sigma from model 0's variance only, util_functions.py:163-167, :233): model 1 runs
    the mean-only kernel first, model 0's launch carries the acquisition.  Against the unfused sequence (both models
    through the full kernel, whose FP32 mean of model 1 is summed in another order: 1e-6 of the scale) and against
    the FP64 path."""
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    X, Y, ells, sf2 = make_problem(n, d)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    spec = ob.spec_ehvi(r, PF, ob.host_prep.cached_samples(2, 5, seed=0), "reference")
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=3)
    before = _cabi.Context.get(0).launch_count()
    fused = ob.score(models, spec, pool, precision="fast", want_acq=True)
    n_fused = _cabi.Context.get(0).launch_count() - before
    plain = ob.score(models, spec, pool, precision="fast", want_acq=True, want_posterior=True)
    n_plain = _cabi.Context.get(0).launch_count() - before - n_fused
    only = ob.score(models, spec, pool, precision="fast")
    assert n_fused < n_plain
    a_f, a_p = fused.acq.cpu().numpy(), plain.acq.cpu().numpy()
    np.testing.assert_allclose(a_f, a_p, rtol=1e-4, atol=1e-5 * np.abs(a_p).max())
    assert (fused.best_index, fused.best_value) == (only.best_index, only.best_value)
    assert fused.best_value == a_f[fused.best_index] == np.nanmax(a_f)
    a_r = ob.score(models, spec, pool, precision="fp64", want_acq=True).acq.cpu().numpy()
    np.testing.assert_allclose(a_f, a_r, rtol=5e-3, atol=2e-3 * np.abs(a_r).max())


@pytest.mark.parametrize("P", [368, 380, 1000])
def test_fused_acquisition_shared_memory_budget(P):
    """The fused epilogue keeps the front's stripes beside the operand rings.  At d = 12 about 3 KB are free: P = 368
    fits together with the step schedule, P = 380 only with the schedule left in global memory, P = 1000 not at all
    (the unfused sequence runs).  Same results in all three cases."""
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    n, d, m = 1024, 12, 4096
    X, Y, ells, sf2 = make_problem(n, d)
    t = np.linspace(0.0, 1.0, P)
    Yf = np.column_stack([t, 1.0 - t])                     # P points on the first front ...
    Yd = 1.5 + 0.1 * np.abs(Y[: n - P] / np.abs(Y).max())  # ... the rest dominated by all of them
    Y2 = np.vstack([Yf, Yd]) + 1e-7 * Y
    models = [ob.GPModel(X, Y2[:, i], ells[i], sf2[i], device=DEV) for i in range(2)]
    PF, r = ob.host_prep.calc_pf(Y2), Y2.max(0) + 0.1
    assert len(PF) == P
    spec = ob.spec_ehvi(r, PF, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=3)
    before = _cabi.Context.get(0).launch_count()
    a = ob.score(models, spec, pool, precision="fast", want_acq=True)
    n_a = _cabi.Context.get(0).launch_count() - before
    b = ob.score(models, spec, pool, precision="fast", want_acq=True, want_posterior=True)
    n_b = _cabi.Context.get(0).launch_count() - before - n_a
    if all(g.plane_format == "f8c" for g in models):
        assert (n_a < n_b) == (P < 384)                    # fused exactly while the stripes fit
    np.testing.assert_array_equal(a.acq.cpu().numpy(), b.acq.cpu().numpy())
    assert (a.best_index, a.best_value) == (b.best_index, b.best_value)


# ------------------------------------------------------------------------------------------
# section 8f-1: marginal likelihood + gradient on the device (hyper-parameter fit)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kernel", [(40, 2, "matern52"), (200, 5, "matern52"), (130, 3, "rbf"), (600, 10, "matern52")])
def test_device_nlml_and_gradient_match_host(n, d, kernel):
    import ctypes as C
    from optimobo_b200.fit import _nlml_and_grad
    from optimobo_b200.gp import _KERNELS, current_stream_ptr
    rng = np.random.default_rng(n)
    X = rng.random((n, d)); y = np.sin(3 * X[:, 0]) + X[:, -1] ** 2 + 0.1 * rng.normal(size=n)
    theta = np.concatenate(([0.3], rng.uniform(-0.4, 0.5, d)))
    f_host, g_host = _nlml_and_grad(theta, X, y, kernel, 1e-8)
    dev = torch.device(DEV)
    Xd, yd = torch.as_tensor(X).to(dev), torch.as_tensor(y).to(dev)
    state = torch.empty(_cabi.state_bytes(n, d), dtype=torch.uint8, device=dev)
    ell = (C.c_double * d)(*np.exp(theta[1:]).tolist())
    spec = _cabi.GpSpec(n=n, d=d, kernel=_KERNELS[kernel], reserved=0, sigma_f2=float(np.exp(theta[0])), sigma_n2=0.0,
                        jitter=1e-8, X=Xd.data_ptr(), y=yd.data_ptr(), ell=ell)
    out = (C.c_double * (d + 2))()
    _cabi.check(_cabi.lib().ombo_gp_nlml_grad(_cabi.Context.get(0).handle, C.byref(spec), C.c_void_p(state.data_ptr()),
                                              out, current_stream_ptr(dev)))
    v = np.frombuffer(out, dtype=np.float64, count=d + 2)
    np.testing.assert_allclose(v[0], f_host, rtol=1e-8, atol=1e-6)
    np.testing.assert_allclose(v[1:], g_host, rtol=1e-5, atol=1e-6 * np.abs(g_host).max())


def test_device_fit_reaches_the_host_optimum():
    from optimobo_b200.fit import _nlml_and_grad, fit_hyperparameters, fit_hyperparameters_device
    rng = np.random.default_rng(4)
    X = rng.random((80, 3)); y = np.cos(4 * X[:, 0]) * X[:, 1] + X[:, 2]
    ell_d, sf2_d = fit_hyperparameters_device(X, y, device=DEV)
    ell_h, sf2_h = fit_hyperparameters(X, y)
    f_d = _nlml_and_grad(np.log(np.concatenate(([sf2_d], ell_d))), X, y, "matern52", 1e-8)[0]
    f_h = _nlml_and_grad(np.log(np.concatenate(([sf2_h], ell_h))), X, y, "matern52", 1e-8)[0]
    assert abs(f_d - f_h) <= 1e-3 * abs(f_h) + 1e-3


# ------------------------------------------------------------------------------------------
# SURVEY section 8f rank 2: candidate-independent prep on the device
# (first front, exact 2-D / 3-D hypervolume, 2-D cell decomposition)
# ------------------------------------------------------------------------------------------
def test_device_prep_anchors():
    """Hand-checkable values of SURVEY section 8c."""
    front = np.array([[.1, .9], [.4, .5], [.8, .2]])
    assert ob.device_prep.hypervolume(front, [1, 1], DEV) == pytest.approx(0.39, abs=1e-15)
    cells = ob.device_prep.decompose_into_cells(front, [0, 0], [1, 1], DEV).cpu().numpy()
    want = np.array([[[.1, 1], [0, 0]], [[.4, .9], [.1, 0]], [[.8, .5], [.4, 0]], [[1, .2], [.8, 0]]])
    np.testing.assert_array_equal(cells, want)
    assert ob.device_prep.hypervolume(np.zeros((0, 2)), [1, 1], DEV) == 0.0
    assert ob.device_prep.hypervolume([[2.0, 0.5]], [1, 1], DEV) == 0.0           # beyond the reference point
    assert ob.device_prep.hypervolume([[0.25, 0.5, 0.5]], [1, 1, 1], DEV) == pytest.approx(0.75 * 0.5 * 0.5)


@pytest.mark.parametrize("n,k", [(1, 2), (2, 2), (57, 2), (300, 3), (1024, 2), (1500, 3), (4096, 2), (700, 5)])
def test_device_pareto_front_matches_host_and_oracle(n, k):
    rng = np.random.default_rng(n + k)
    Y = rng.random((n, k))
    Y[rng.integers(0, n, n // 8)] = Y[rng.integers(0, n, n // 8)]     # exact duplicates
    Y[:, 0] = np.round(Y[:, 0], 2)                                     # ties in one objective
    mask = ob.device_prep.pareto_mask(Y, DEV).cpu().numpy()
    np.testing.assert_array_equal(mask, ob.host_prep.pareto_mask(Y))
    np.testing.assert_array_equal(ob.device_prep.calc_pf(Y, DEV), O.calc_pf(Y))


@pytest.mark.parametrize("n,k", [(5, 2), (120, 2), (1024, 2), (3000, 2), (40, 3), (400, 3), (1024, 3)])
def test_device_hypervolume_matches_host_and_oracle(n, k):
    rng = np.random.default_rng(10 * n + k)
    Y = rng.random((n, k)) ** 2
    Y[: n // 10] = Y[n // 10: 2 * (n // 10)]                            # duplicates
    Y[:, -1] = np.round(Y[:, -1], 2)                                    # ties in the slicing objective
    ref = np.full(k, 0.9)                                               # some points beyond the reference point
    hv = ob.device_prep.hypervolume(Y, ref, DEV)
    assert hv == ob.host_prep.hypervolume(Y, ref)                       # same order of operations: bit-identical
    assert hv == pytest.approx(O.hypervolume(Y, ref), rel=1e-12)
    # size-independent property: hypervolume of the whole sample = hypervolume of its first front
    assert hv == pytest.approx(ob.device_prep.hypervolume(ob.device_prep.calc_pf(Y, DEV), ref, DEV), rel=1e-12)


@pytest.mark.parametrize("n", [1, 2, 33, 500])
def test_device_cells_match_host_oracle_and_feed_hv_poi(n):
    rng = np.random.default_rng(n)
    Y = rng.random((max(n * 6, 4), 2))
    pf = ob.host_prep.calc_pf(Y)[:n] if n > 1 else Y[:1]
    ideal, maxp = np.array([-0.1, -0.2]), np.array([1.1, 1.3])
    cells = ob.device_prep.decompose_into_cells(pf, ideal, maxp, DEV)
    np.testing.assert_array_equal(cells.cpu().numpy(), ob.host_prep.decompose_into_cells(pf, ideal, maxp))
    np.testing.assert_array_equal(cells.cpu().numpy(), O.decompose_into_cells_2d(pf, ideal, maxp))
    # the device cells drive the EMO acquisition exactly like the host ones
    m = 257
    mu, var = rng.random((2, m)), 0.01 + rng.random((2, m))
    a_dev, _, _ = ob.acquire_from_posterior(ob.spec_hv_poi(cells.cpu().numpy()), mu, var, device=DEV)
    a_ora = O.hv_poi_batched(mu.T, var.T, O.decompose_into_cells_2d(pf, ideal, maxp))
    np.testing.assert_allclose(a_dev.cpu().numpy(), a_ora, rtol=1e-9, atol=1e-300)


# ------------------------------------------------------------------------------------------
# SURVEY section 8f rank 4: joint posterior samples (the device side of TuRBO's Thompson sampling)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,m,S,kernel", [(30, 2, 200, 4, "matern52"), (100, 5, 1000, 3, "matern52"),
                                            (64, 3, 129, 1, "rbf"), (200, 10, 1000, 10, "matern52"),
                                            (257, 4, 63, 5, "matern52")])
def test_joint_posterior_samples_vs_oracle(n, d, m, S, kernel):
    """out = mu + chol(Sigma + diag_add I) Z against the numpy/LAPACK restatement on the same Z.  The
    jitter keeps the m x m covariance comfortably positive definite so that both Cholesky factors
    are well conditioned (rtol 1e-6 of the sample scale)."""
    X, Y, ells, sf2 = make_problem(n, d)
    noise = 1e-4 if kernel == "rbf" else 0.0
    gp = ob.GPModel(X, Y[:, 0], ells[0], sf2[0], noise=noise, kernel=kernel, device=DEV)
    st = O.gp_fit_state(X, Y[:, 0], ells[0], sf2[0], sigma_n2=noise,
                        kernel=O.KERNEL_RBF if kernel == "rbf" else O.KERNEL_MATERN52, form="direct")
    rng = np.random.default_rng(n + m)
    Xc = rng.random((m, d))
    Z = rng.standard_normal((m, S))
    jitter = 1e-6 * sf2[0]
    got = gp.posterior_samples_from(Xc, Z, jitter=jitter)
    assert got.shape == (m, 1, S) and gp.sample_jitter == jitter
    want = O.posterior_samples(st, Xc, Z, noise + jitter)
    scale = np.abs(want).max()
    np.testing.assert_allclose(got[:, 0, :], want, rtol=1e-6, atol=2e-6 * scale)
    # Z = 0 returns the posterior mean of the scoring path
    mu = gp.posterior_samples_from(Xc, np.zeros((m, 1)), jitter=jitter)[:, 0, 0]
    mu_ref, _ = ob.posterior([gp], Xc)
    np.testing.assert_allclose(mu, mu_ref[0].cpu().numpy(), rtol=1e-9, atol=1e-9 * max(1.0, np.abs(mu).max()))


def test_joint_posterior_samples_statistics_and_jitter_retry():
    """Distributional check (what the reference's np.random.multivariate_normal draw shares with the
    Cholesky draw): sample mean -> mu, sample variance -> diag(Sigma); and duplicate candidates
    (singular covariance) are handled by the jitchol-style retry."""
    n, d, m, S = 60, 3, 150, 4000
    X, Y, ells, sf2 = make_problem(n, d)
    gp = ob.GPModel(X, Y[:, 1], ells[1], sf2[1], device=DEV)
    st = O.gp_fit_state(X, Y[:, 1], ells[1], sf2[1], form="direct")
    Xc = np.random.default_rng(1).random((m, d))
    smp = gp.posterior_samples(Xc, size=S, rng=np.random.default_rng(2))[:, 0, :]
    mu, Sig = O.gp_posterior_joint(st, Xc)
    sd = np.sqrt(np.diag(Sig))
    assert np.abs(smp.mean(1) - mu).max() < 6 * sd.max() / np.sqrt(S)
    np.testing.assert_allclose(smp.std(1), sd, rtol=0.1, atol=1e-3)
    Xdup = np.vstack((Xc[:40], Xc[:40]))
    out = gp.posterior_samples(Xdup, size=3, rng=np.random.default_rng(3), jitter=0.0)
    assert np.all(np.isfinite(out)) and gp.sample_jitter > 0
    np.testing.assert_allclose(out[:40], out[40:], atol=1e-2 * np.sqrt(sf2[1]))
    with pytest.raises(ValueError):
        gp.posterior_samples_from(Xc[:, :2], np.zeros((m, 1)))


def test_conditioning_proxy_guards_the_fast_mode():
    """GPModel.conditioning = (max L_ii / min L_ii)^2; the optimisers' precision="auto" falls back to FP64
    on large but ill-conditioned GPs, an explicit precision="fast" warns."""
    import warnings
    from optimobo_b200.algorithms.base import PoolOptimiserBase
    from optimobo_b200.problem import Problem
    rng = np.random.default_rng(0)
    good_X, bad_X = rng.random((400, 10)), rng.random((400, 2))
    y = np.sin(3 * good_X.sum(1))
    good = ob.GPModel(good_X, y, 0.7 * np.ones(10), 1.5, device=DEV)
    bad = ob.GPModel(bad_X, y, 0.3 * np.ones(2), 1.5, device=DEV)
    for gp, X, ell in ((good, good_X, 0.7), (bad, bad_X, 0.3)):
        dg = np.diag(O.gp_fit_state(X, y, ell * np.ones(X.shape[1]), 1.5, form="direct")["L"])
        assert gp.conditioning == pytest.approx((dg.max() / dg.min()) ** 2, rel=1e-6)
    assert good.conditioning < ob.GPModel.FAST_MODE_CONDITIONING_LIMIT < bad.conditioning
    base = PoolOptimiserBase(Problem(n_var=10, n_obj=2, xl=np.zeros(10), xu=np.ones(10)), device=DEV)
    if _cabi.fast_path_available():
        assert base._precision_for([good]) == "fast" and base._precision_for([bad]) == "fp64"
        mid = ob.GPModel(good_X[:200], y[:200], 0.7 * np.ones(10), 1.5, device=DEV)      # C2-sized: fast as well
        tiny = ob.GPModel(good_X[:40], y[:40], 0.7 * np.ones(10), 1.5, device=DEV)       # tiny: FP64 is cheap
        assert base._precision_for([mid]) == "fast" and base._precision_for([tiny]) == "fp64"
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            ob.posterior([good], good_X[:10], precision="fast")
            assert not [x for x in w if issubclass(x.category, RuntimeWarning)]
            ob.posterior([bad], bad_X[:10], precision="fast")
            assert [x for x in w if issubclass(x.category, RuntimeWarning)]


def test_fast_mode_operand_format_follows_conditioning():
    """K3 chooses the operand format of the fast mode from the conditioning proxy: "f8c" (fp16 plane + two e4m3
    correction planes, the CTA-pair kernel) up to kappa = 100, scaled fp16 x3 planes (+ direct-difference distances)
    beyond; with OMBO_NO_F8C the well-conditioned GPs get bf16 x3 planes.  Every instantiation meets the tolerance
    inside the guarded range."""
    if not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    rng = np.random.default_rng(5)
    seen = set()
    for n, d, ell in ((600, 10, 0.7), (600, 6, 0.6), (1024, 5, 0.5), (700, 10, 1.5)):
        X = rng.random((n, d))
        y = np.sin(3 * X.sum(1))
        gp = ob.GPModel(X, y, ell * np.ones(d), 1.5, device=DEV)
        assert gp._flags == (2 if gp.conditioning > 100.0 else 4)
        assert gp.plane_format == ("fp16x3" if gp.conditioning > 100.0 else "f8c")
        seen.add(gp._flags)
        assert gp.conditioning < ob.GPModel.FAST_MODE_CONDITIONING_LIMIT
        Xc = rng.random((3000, d))
        st = O.gp_fit_state(X, y, ell * np.ones(d), 1.5, form="direct")
        mu_o, var_o = O.gp_posterior(st, Xc)
        mu, var = ob.posterior([gp], Xc, precision="fast")
        np.testing.assert_allclose(mu[0].cpu().numpy(), mu_o, rtol=1e-3, atol=1e-3 * max(1.0, np.abs(mu_o).max()))
        np.testing.assert_allclose(np.sqrt(var[0].cpu().numpy()), np.sqrt(var_o), rtol=1e-3, atol=1e-3 * np.sqrt(1.5))
    assert seen == {2, 4}
    # d > 12 has no f8c instantiation: bf16 x3 planes
    X = rng.random((300, 16))
    gp = ob.GPModel(X, np.sin(X.sum(1)), 2.0 * np.ones(16), 1.0, device=DEV)
    assert gp.plane_format == ("fp16x3" if gp.conditioning > 100.0 else "bf16x3")
