"""GPU: the exact k-objective EHVI over the box decomposition (OMBO_ACQ_EHVI_BOX, k_acquire_box) against the grid
oracle, in both precisions, through the whole scoring path and the optimiser."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi, distributed  # noqa: E402
from optimobo_b200.algorithms import MultiSurrogateOptimiser  # noqa: E402
from optimobo_b200.problem import Problem  # noqa: E402
from oracle import oracle as O  # noqa: E402
from ehvi_oracle import ehvi_grid_batched, expected_shortfall  # noqa: E402
from test_gpu_parity import _check_selection  # noqa: E402

DEV = "cuda:0"
needs_fast = pytest.mark.skipif(not _cabi.fast_path_available(), reason="fast path not built")


def _sphere(P, k, rng, offset=0.0):
    X = np.abs(rng.normal(size=(P, k)))
    return offset + X / np.linalg.norm(X, axis=1, keepdims=True)


def _posteriors(PF, m, rng, spread=0.05, sd=0.05):
    """m posteriors near the front: a front point + N(0, spread^2), sigma ~ U(0.5, 1.5) * sd."""
    k = PF.shape[1]
    mu = PF[rng.integers(0, len(PF), m)] + rng.normal(0, spread, size=(m, k))
    var = (sd * rng.uniform(0.5, 1.5, size=(m, k))) ** 2
    return mu, var


def _acquire(spec, mu, var, index_base=0):
    acq, bv, bi = ob.acquire_from_posterior(spec, mu.T, var.T, DEV, index_base=index_base)
    return acq.cpu().numpy(), bv, bi


def _box_sum(spec, mu, var):
    """numpy sum over the spec's own boxes (checked against the grid oracle on the CPU)."""
    table, boxes = spec.stripes, spec.cells.astype(np.int64)
    sd = np.sqrt(var)
    out = np.ones((len(mu), len(boxes)))
    for i in range(table.shape[0]):
        U, L = table[i, boxes[:, 0, i]], table[i, boxes[:, 1, i]]
        out *= (expected_shortfall(U[None, :], mu[:, i:i + 1], sd[:, i:i + 1])
                - expected_shortfall(L[None, :], mu[:, i:i + 1], sd[:, i:i + 1]))
    return out.sum(1)


# ------------------------------------------------------------------------------------------
# K4 alone
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,P", [(2, 40), (3, 66), (3, 150), (4, 30)])
def test_device_vs_grid_oracle_fp64(k, P):
    rng = np.random.default_rng(k * 100 + P)
    PF = _sphere(P, k, rng)
    r = PF.max(0) + 0.1
    mu, var = _posteriors(PF, 3000, rng)
    mu[:10] = PF.min(0) - 1.0                                  # far below the front: both breakpoints above the mean
    mu[10:20] = r + 1.0                                        # beyond r
    got, bv, bi = _acquire(ob.spec_ehvi_box(r, PF), mu, var)
    want = ehvi_grid_batched(mu, var, PF, r)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-14 * np.abs(want).max())
    assert bi == O.argmax_lowest_index(got) and bv == got[bi]


def test_k2_equals_exact_ehvi2d(golden):
    mu, var = golden["acq_in_mu2"], golden["acq_in_var2"]
    PF, r = golden["acq_out_calc_pf"], golden["acq_in_ref"]
    box, _, _ = _acquire(ob.spec_ehvi_box(r, PF), mu, var)
    exact, _, _ = ob.acquire_from_posterior(ob.spec_ehvi(r, PF, golden["acq_in_cache2"], semantics="exact"),
                                            mu.T, var.T, DEV)
    exact = exact.cpu().numpy()
    np.testing.assert_allclose(box, exact, rtol=1e-12, atol=1e-12 * np.abs(exact).max())


@pytest.mark.parametrize("m", [1, 255, 257, 5001])
def test_ragged_m_index_base_and_reproducibility(m):
    rng = np.random.default_rng(m)
    PF = _sphere(50, 3, rng)
    r = PF.max(0) + 0.1
    mu, var = _posteriors(PF, m, rng)
    spec = ob.spec_ehvi_box(r, PF)
    base = 10 ** 9 + 17
    got, bv, bi = _acquire(spec, mu, var, index_base=base)
    np.testing.assert_allclose(got, ehvi_grid_batched(mu, var, PF, r), rtol=1e-9, atol=1e-14)
    assert bi == base + O.argmax_lowest_index(got) and bv == got[bi - base]
    again, bv2, bi2 = _acquire(spec, mu, var, index_base=base)
    assert np.array_equal(got, again) and (bv2, bi2) == (bv, bi)


# ------------------------------------------------------------------------------------------
# whole path at the C4 shape: DTLZ2, n = 512, d = 12, k = 3
# ------------------------------------------------------------------------------------------
def _c4(n=512, d=12):
    rng = np.random.default_rng(4)
    X = rng.random((n, d))
    g = ((X[:, 2:] - .5) ** 2).sum(1)
    a, b = .5 * np.pi * X[:, 0], .5 * np.pi * X[:, 1]
    Y = np.column_stack([(1 + g) * np.cos(a) * np.cos(b), (1 + g) * np.cos(a) * np.sin(b), (1 + g) * np.sin(a)])
    ells = [(0.7 + 0.1 * i) * np.ones(d) * (1 + 0.05 * np.arange(d)) for i in range(3)]
    sf2 = [1.0 + i for i in range(3)]
    return X, Y, ells, sf2


@pytest.fixture(scope="module")
def c4():
    X, Y, ells, sf2 = _c4()
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(3)]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0) + 0.1
    return X, Y, ells, sf2, models, ob.spec_ehvi_box(r, PF), PF, r


@pytest.mark.parametrize("precision", ["fp64", pytest.param("fast", marks=needs_fast)])
def test_full_path_c4(c4, precision):
    X, Y, ells, sf2, models, spec, PF, r = c4
    m, d = 1 << 12, X.shape[1]
    lo, hi = np.zeros(d), np.ones(d)
    pool = ob.CandidatePool.counter(m, lo, hi, seed=2)
    Xc = O.candidates_from_counter(2, 0, m, lo, hi)
    post = [O.gp_posterior(O.gp_fit_state(X, Y[:, i], ells[i], sf2[i]), Xc) for i in range(3)]
    mu_o, var_o = np.array([p[0] for p in post]).T, np.array([p[1] for p in post]).T
    want = ehvi_grid_batched(mu_o, var_o, PF, r)
    res = ob.score(models, spec, pool, precision=precision, want_acq=True)
    got = res.acq.cpu().numpy()
    # the posterior's tolerance carries over: FP64 rtol 1e-6 on sigma, the fast mode 1e-3
    tol = 1e-5 if precision == "fp64" else 2e-3
    np.testing.assert_allclose(got, want, rtol=tol, atol=tol * np.abs(want).max())
    _check_selection(got, want, res.best_index, rtol=1e-6 if precision == "fp64" else 1e-3)
    x, neg, idx = ob.propose(models, spec, pool, precision=precision)
    assert idx == res.best_index and np.array_equal(x, Xc[idx]) and neg == -res.best_value


@needs_fast
@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_fp32_kernel_vs_grid_oracle(offset):
    """The FP32 K4 of the fast mode on the fast path's own posteriors: within 1e-3 of the scale against the grid
    oracle, and each value within 2e-5 of the FP64 kernel's on the same posteriors.  offset = 1e3 moves the front (unit
    spread) far above the means, so t - mu ~ 1e3 must keep the digits of breakpoint spacings ~ 1e-2."""
    X, Y, ells, sf2 = _c4(n=256, d=6)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(3)]
    PF = ob.host_prep.calc_pf(Y) + offset
    r = PF.max(0) + 0.1
    spec = ob.spec_ehvi_box(r, PF)
    pool = ob.CandidatePool.counter(1 << 12, np.zeros(6), np.ones(6), seed=5)
    res = ob.score(models, spec, pool, precision="fast", want_posterior=True, want_acq=True)
    mu, var = res.mu.cpu().numpy().T, res.var.cpu().numpy().T
    want = ehvi_grid_batched(mu, var, PF, r)
    got = res.acq.cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-3 * np.abs(want).max())
    # the same posteriors through the FP64 kernel
    f64, _, _ = _acquire(spec, mu, var)
    np.testing.assert_allclose(f64, want, rtol=1e-9, atol=1e-12 * np.abs(want).max())
    big = np.abs(f64) > 1e-3 * np.abs(f64).max()
    np.testing.assert_allclose(got[big], f64[big], rtol=2e-5)
    np.testing.assert_allclose(got, f64, rtol=0, atol=2e-6 * np.abs(f64).max())


def test_any_spec_entries_take_the_box_kind(c4):
    """propose / polish / top_candidates / distributed.score_sharded need no change for the new kind."""
    X, Y, ells, sf2, models, spec, PF, r = c4
    d = X.shape[1]
    pool = ob.CandidatePool.counter(1 << 20, np.zeros(d), np.ones(d), seed=9)
    whole = ob.score(models, spec, pool)
    shards = [ob.score(models, spec, pool.shard(q, 4)) for q in range(4)]
    best = max(shards, key=lambda s: (s.best_value, -s.best_index))
    assert (best.best_value, best.best_index) == (whole.best_value, whole.best_index)
    assert distributed.score_sharded(models, spec, pool) == (whole.best_value, whole.best_index)
    rows, vals = ob.top_candidates(models, spec, pool, 4, head=1 << 14)
    assert rows.shape == (4, d) and np.all(np.diff(vals) <= 0)
    np.testing.assert_allclose(ob.evaluate(models, spec, rows), vals, rtol=1e-9)
    xp, vp, per = ob.polish(models, spec, rows[:2], np.zeros(d), np.ones(d), max_iter=5)
    assert vp >= vals[0] * (1 - 1e-9) and per.shape == (2,)
    x, neg, idx = ob.propose(models, spec, pool, refine_rounds=1, refine_candidates=1 << 12)
    assert -neg >= whole.best_value and x.shape == (d,)
    np.testing.assert_allclose(ob.EHVI_box(x, models, r, PF), [-neg], rtol=1e-9)


# ------------------------------------------------------------------------------------------
# size limits
# ------------------------------------------------------------------------------------------
def test_largest_front_scores_and_one_more_raises():
    rng = np.random.default_rng(3)
    P = _cabi.EHVI_BOX_MAX_BREAKS - 2
    F = _sphere(4 * P, 3, rng)
    F = ob.host_prep.calc_pf(F)[:P]
    assert len(F) == P
    r = F.max(0) + 0.1
    spec = ob.spec_ehvi_box(r, F)
    assert spec.stripes.shape[1] == _cabi.EHVI_BOX_MAX_BREAKS
    mu, var = _posteriors(F, 2000, rng)
    got, _, _ = _acquire(spec, mu, var)
    np.testing.assert_allclose(got[:64], _box_sum(spec, mu[:64], var[:64]), rtol=1e-9, atol=1e-14)
    # k = 4 at the largest B: 512 points on a 2-D line of a 4-D front (few boxes, the widest table)
    t = np.linspace(0, 1, P)
    F4 = np.column_stack([t, 1 - t, np.full(P, 0.5), np.full(P, 0.5)])
    spec4 = ob.spec_ehvi_box(np.full(4, 1.1), F4)
    assert spec4.stripes.shape[1] == _cabi.EHVI_BOX_MAX_BREAKS
    mu4, var4 = _posteriors(F4, 1000, rng)
    got4, _, _ = _acquire(spec4, mu4, var4)
    np.testing.assert_allclose(got4, _box_sum(spec4, mu4, var4), rtol=1e-9, atol=1e-14)
    # one point more: a clean error, no launch
    G = _sphere(4 * (P + 1), 3, np.random.default_rng(4))
    G = ob.host_prep.calc_pf(G)[:P + 1]
    with pytest.raises(_cabi.OmboError, match="breakpoints"):
        _acquire(ob.spec_ehvi_box(G.max(0) + 0.1, G), mu, var)
    big = ob.AcquisitionSpec(kind=_cabi.ACQ_EHVI_BOX, n_obj=3, ref=tuple(r), stripes=spec.stripes,
                             cells=np.ones((_cabi.EHVI_BOX_MAX_BOXES + 1, 2, 3)), n_models=3)
    with pytest.raises(_cabi.OmboError, match="boxes"):
        _acquire(big, mu, var)


@needs_fast
def test_largest_front_fast():
    rng = np.random.default_rng(6)
    P = _cabi.EHVI_BOX_MAX_BREAKS - 2
    X, Y, ells, sf2 = _c4(n=256, d=6)
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(3)]
    F = ob.host_prep.calc_pf(_sphere(4 * P, 3, rng))[:P]
    spec = ob.spec_ehvi_box(F.max(0) + 0.1, F)
    res = ob.score(models, spec, ob.CandidatePool.counter(256, np.zeros(6), np.ones(6), seed=3), precision="fast",
                   want_posterior=True, want_acq=True)
    mu, var = res.mu.cpu().numpy().T, res.var.cpu().numpy().T
    want = _box_sum(spec, mu, var)
    np.testing.assert_allclose(res.acq.cpu().numpy(), want, rtol=1e-3, atol=1e-3 * np.abs(want).max())


# ------------------------------------------------------------------------------------------
# optimiser
# ------------------------------------------------------------------------------------------
class DTLZ2(Problem):
    def __init__(self, n_var=6, n_obj=3):
        super().__init__(n_var=n_var, n_obj=n_obj, xl=np.zeros(n_var), xu=np.ones(n_var))

    def _evaluate(self, x, out, *args, **kwargs):
        g = ((x[:, 2:] - 0.5) ** 2).sum(1)
        a, b = 0.5 * np.pi * x[:, 0], 0.5 * np.pi * x[:, 1]
        F = [(1 + g) * np.cos(a) * np.cos(b), (1 + g) * np.cos(a) * np.sin(b), (1 + g) * np.sin(a)]
        out["F"] = F[:1] + [(1 + g) * np.sin(a)] if self.n_obj == 2 else F


class _Recording(MultiSurrogateOptimiser):
    def _propose(self, models, spec):
        x, neg = super()._propose(models, spec)
        self.seen = getattr(self, "seen", []) + [(spec.kind, -neg)]
        return x, neg


@pytest.mark.parametrize("n_obj", [3, 2])
def test_optimiser_box(n_obj):
    opt = _Recording(DTLZ2(n_obj=n_obj), ehvi="box", n_candidates=1 << 14, seed=0, device=DEV, max_f_eval=200)
    res = opt.solve(budget=3, n_init_samples=12)
    assert res.ysample.shape == (15, n_obj) and np.all(np.isfinite(res.ysample))
    assert [kind for kind, _ in opt.seen] == [_cabi.ACQ_EHVI_BOX] * 3
    assert max(v for _, v in opt.seen) > 0
    with pytest.raises(ValueError):
        MultiSurrogateOptimiser(DTLZ2(), ehvi="grid")
