"""GPU: Kriging-believer batches (propose_batch) select what a brute-force Kriging believer selects -- q full passes
with the fantasy models, the best candidate not selected yet at each step -- with and without the shortlist
certificate, and the optimisers' batch_size surface evaluates exactly n_init + budget points."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi  # noqa: E402
from optimobo_b200.acquisition import _CERT_TAU  # noqa: E402
from optimobo_b200.algorithms import MonoSurrogateOptimiser, MultiSurrogateOptimiser  # noqa: E402
from optimobo_b200.problem import ElementwiseProblem  # noqa: E402

DEV = "cuda:0"
pytestmark = pytest.mark.gpu
FAST = ["fp64", "fast"] if _cabi.fast_path_available() else ["fp64"]


def zdt(n, d, seed=0, k=2):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    f1 = X[:, 0]
    g = 1 + 9.0 / (d - 1) * X[:, 1:].sum(1)
    cols = [f1, g * (1 - np.sqrt(f1 / g)), g * (1 - X[:, 1]) + 0.5 * f1][:k]
    return X, np.column_stack(cols)


def workload(kind):
    """(models, spec_for, d): C5-shaped 2-D EHVI (n = 1024), C4-like box EHVI of 3 objectives, C2-shaped EI."""
    if kind == "ei":
        X, Y = zdt(256, 10)
        model = ob.GPModel(X, Y[:, 1], 0.8 * np.ones(10), 2.0, device=DEV)
        best = float(Y[:, 1].min())
        return [model], lambda Yb: ob.spec_ei(min(best, float(Yb.min())) if len(Yb) else best), 10
    if kind == "box3":
        X, Y = zdt(512, 8, k=3)
        models = [ob.GPModel(X, Y[:, i], [0.7, 0.8, 0.9][i] * np.ones(8), [1.0, 2.0, 1.5][i], device=DEV)
                  for i in range(3)]
        PF, r = ob.host_prep.calc_pf(Y), Y.max(0)

        def spec_for(Yb):
            inside = Yb[np.all(Yb <= r, axis=1)] if len(Yb) else Yb
            return ob.spec_ehvi_box(r, ob.host_prep.calc_pf(np.vstack([PF, inside])) if len(inside) else PF)
        return models, spec_for, 8
    X, Y = zdt(1024, 10)
    models = [ob.GPModel(X, Y[:, i], [0.7, 0.8][i] * np.ones(10), [1.0, 2.0][i], device=DEV) for i in range(2)]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    sem = "exact" if kind == "ehvi_exact" else "reference"

    def spec_for(Yb):
        inside = Yb[np.all(Yb <= r, axis=1)] if len(Yb) else Yb
        return ob.spec_ehvi(r, ob.host_prep.calc_pf(np.vstack([PF, inside])) if len(inside) else PF, cache, sem)
    return models, spec_for, 10


def brute_force(models, spec_for, pool, q, precision):
    """q full passes with the fantasy models; per step the pick, its value and the top-two gap of the non-selected."""
    Yb = np.empty((0, len(models)))
    picked, gaps, scales = [], [], []
    for j in range(q):
        if j > 0:
            x = pool.rows(picked[-1], 1, DEV)
            mu, _ = ob.posterior(models, x, precision="fp64")
            y = mu[:, 0].cpu().numpy()
            Yb = np.vstack([Yb, y[None, :]])
            models = [m.with_observations(x, y[g:g + 1]) for g, m in enumerate(models)]
        acq = ob.score(models, spec_for(Yb), pool, precision=precision, want_acq=True, want_best=False).acq
        a = np.where(np.isnan(acq.cpu().numpy()), -np.inf, acq.cpu().numpy())
        a[np.asarray(picked, dtype=np.int64) - pool.index_base] = -np.inf
        order = np.argsort(-a, kind="stable")
        picked.append(int(order[0]) + pool.index_base)
        gaps.append(a[order[0]] - a[order[1]])
        scales.append(abs(a[order[0]]))
    return picked, gaps, scales


def same_selection(got, want, gaps, scales, tau):
    """Identical picks, except that a step whose brute-force top-two gap is within tau * scale may differ (and every
    later step then conditions on another point)."""
    for j, (g, w) in enumerate(zip(got, want)):
        if g != w:
            assert gaps[j] <= tau * max(scales[j], 1e-300), (j, got, want)
            return


CASES = [("ei", p) for p in FAST] + [("ehvi_exact", p) for p in FAST] + [("ehvi_ref", "fp64"), ("box3", "fp64")]


@pytest.mark.parametrize("kind,precision", CASES)
@pytest.mark.parametrize("shortlist", [64, 4096])
def test_batch_matches_brute_force_believer(kind, precision, shortlist):
    models, spec_for, d = workload(kind)
    m = 1 << 16 if kind == "box3" else 1 << 18
    pool = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=11)
    q = 4
    X, neg, idx, cert = ob.propose_batch(models, spec_for, pool, q, precision=precision, shortlist=shortlist)
    assert X.shape == (q, d) and neg.shape == (q,) and cert.dtype == bool
    assert len(set(idx.tolist())) == q
    np.testing.assert_array_equal(X, pool.rows(0, m, DEV).cpu().numpy()[idx])
    want, gaps, scales = brute_force(models, spec_for, pool, q, precision)
    same_selection(list(idx), want, gaps, scales, _CERT_TAU[precision])
    assert not cert[0]
    if kind == "ehvi_ref":
        assert not cert.any()
    # step 0 is propose(refine_rounds=0)'s winner
    _, neg0, i0 = ob.propose(models, spec_for(np.empty((0, len(models)))), pool, precision=precision)
    assert (int(idx[0]), float(neg[0])) == (i0, neg0)


def test_with_observations_does_not_mutate():
    X, Y = zdt(64, 4)
    m = ob.GPModel(X, Y[:, 0], 0.5 * np.ones(4), 1.0, device=DEV)
    X0, y0 = m.X.clone(), m.y.clone()
    m2 = m.with_observations(X[:2] + 0.01, [0.3, 0.4])
    assert torch.equal(m.X, X0) and torch.equal(m.y, y0) and m.n == 64
    assert m2.n == 66 and m2.noise == m.noise and np.array_equal(m2.lengthscale, m.lengthscale)
    Xc = np.random.default_rng(1).random((500, 4))
    mu, var = ob.posterior([m], Xc)
    x1 = torch.as_tensor(Xc[:1], device=DEV)
    mu1 = ob.posterior([m], x1)[0][0].cpu().numpy()
    mu2, var2 = ob.posterior([m.with_observations(x1, mu1)], Xc)
    np.testing.assert_allclose(mu2.cpu().numpy(), mu.cpu().numpy(), rtol=1e-6, atol=1e-6)
    assert bool((var2 <= var * (1 + 1e-6) + 1e-12).all())


class MyProblem(ElementwiseProblem):     # INTEGRATION.md's example
    def __init__(self):
        super().__init__(n_var=2, n_obj=2, xl=np.array([-2, -2]), xu=np.array([2, 2]))

    def _evaluate(self, x, out, *args, **kwargs):
        out["F"] = [100 * (x[0] ** 2 + x[1] ** 2), (x[0] - 1) ** 2 + x[1] ** 2]


KW = dict(n_candidates=1 << 14, seed=0, device="cuda:0", max_f_eval=200)


@pytest.mark.parametrize("acq", ["ehvi", "box", "decomposition"])
def test_multi_optimiser_batches(acq):
    kw = dict(KW, ehvi="box") if acq == "box" else KW
    opt = MultiSurrogateOptimiser(MyProblem(), [0, 0], [700, 12], batch_size=3, **kw)
    func = ob.scalarisations.Tchebicheff([0, 0], [700, 12]) if acq == "decomposition" else None
    res = opt.solve(budget=7, n_init_samples=6, sample_exponent=3, acquisition_func=func)     # 3 + 3 + 1
    assert res.ysample.shape == (13, 2) and res.Xsample.shape == (13, 2)
    assert len(res.hypervolume_convergence) == 3 and len(res.timings) == 3
    assert [t["batch"] for t in res.timings] == [3, 3, 1]
    assert np.all(np.isfinite(res.ysample))


def test_mono_optimiser_batches():
    opt = MonoSurrogateOptimiser(MyProblem(), [0, 0], [700, 12], batch_size=3, **KW)
    res = opt.solve(ob.scalarisations.Tchebicheff([0, 0], [700, 12]), budget=5, n_init_samples=6)   # 3 + 2
    assert res.ysample.shape == (11, 2) and res.Xsample.shape == (11, 2)
    assert len(res.hypervolume_convergence) == 2 and [t["batch"] for t in res.timings] == [3, 2]
