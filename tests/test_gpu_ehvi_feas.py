"""GPU: the constrained box EHVI (OMBO_ACQ_EHVI_BOX_FEAS, k_acquire_box<T, K, true>) -- box EHVI times the
probability that every constraint holds -- against the 50-digit reference, its reduction to the plain box kind, the
FP32 contract in the deep infeasible tail, the whole scoring path, batches and the constrained optimiser."""
import json
import os
import subprocess
import sys

import mpmath as mp
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi, distributed, result  # noqa: E402
from optimobo_b200.algorithms import MultiSurrogateOptimiser  # noqa: E402
from optimobo_b200.problem import Problem  # noqa: E402
from oracle import oracle as O  # noqa: E402
import acq_mpmath as M  # noqa: E402
from test_gpu_batch import brute_force, same_selection  # noqa: E402
from test_gpu_parity import _check_selection  # noqa: E402

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_fast = pytest.mark.skipif(not _cabi.fast_path_available(), reason="fast path not built")
PRECISIONS = ["fp64", pytest.param("fast", marks=needs_fast)]


def _sphere(P, k, rng):
    X = np.abs(rng.normal(size=(P, k)))
    return X / np.linalg.norm(X, axis=1, keepdims=True)


def _pof_mp(mu, var, eps):
    """prod_j Phi(-mu_j / sqrt(var_j + eps)) in 50 digits, per row of mu / var (m, c)."""
    out = []
    for mr, vr in zip(mu, var):
        p = mp.mpf(1)
        for a, b in zip(mr, vr):
            p *= mp.ncdf(-mp.mpf(a) / mp.sqrt(mp.mpf(b) + mp.mpf(eps)))
        out.append(p)
    return out


def _pof64(mu, var, eps):
    from scipy.special import ndtr
    return np.prod(ndtr(-mu / np.sqrt(var + eps)), axis=1)


def _acquire(spec, mu, var, index_base=0):
    acq, bv, bi = ob.acquire_from_posterior(spec, mu.T, var.T, DEV, index_base=index_base)
    return acq.cpu().numpy(), bv, bi


# ------------------------------------------------------------------------------------------
# 1. K4 alone in FP64 against the 50-digit reference
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("front", ["sphere", "empty"])
def test_fp64_against_mpmath(k, front):
    rng = np.random.default_rng(10 * k + (front == "empty"))
    P = {2: 8, 3: 7, 4: 5}[k]
    S = _sphere(P, k, rng)
    r = S.max(0) + 0.1
    if front == "sphere":
        # a duplicate point and two points beyond r (dropped by the decomposition) ride along
        PF = np.vstack([S, S[:1], S[1:2] + np.eye(k)[0] * (r[0] + 1.0), r + 0.5])
    else:
        PF = np.empty((0, k))
    m, c_max = 40, 8 - k
    mu_o = S[rng.integers(0, P, m)] + rng.normal(0, 0.05, size=(m, k))
    var_o = (0.05 * rng.uniform(0.5, 1.5, size=(m, k))) ** 2
    # constraint posteriors from feasible to ~8 sigma infeasible, at sigma of 0.1 to 1
    sd_c = rng.uniform(0.1, 1.0, size=(m, c_max))
    mu_c = sd_c * rng.uniform(-3.0, 8.0, size=(m, c_max))
    var_c = sd_c ** 2
    plain = ob.spec_ehvi_box(r, PF)
    ehvi = M.ehvi_box(plain.stripes, plain.cells, mu_o, var_o)
    for eps in (1e-5, 0.0):
        for c in range(1, c_max + 1):
            spec = ob.spec_ehvi_box_feasible(r, PF, c, var_eps=eps)
            got, bv, bi = _acquire(spec, np.hstack([mu_o, mu_c[:, :c]]), np.hstack([var_o, var_c[:, :c]]))
            want = np.array([float(mp.mpf(e) * p) for e, p in zip(ehvi, _pof_mp(mu_c[:, :c], var_c[:, :c], eps))])
            big = want >= 1e-280
            assert big.sum() >= m // 2
            np.testing.assert_allclose(got[big], want[big], rtol=1e-9, err_msg=f"k={k} c={c} eps={eps}")
            assert np.all(np.abs(got[~big]) < 1e-279) and np.all(got >= 0)
            assert bi == O.argmax_lowest_index(got) and bv == got[bi]


# ------------------------------------------------------------------------------------------
# whole-path fixtures: the C4 shape (DTLZ2, n = 512, d = 12, k = 3) with c = 2 constraint models
# ------------------------------------------------------------------------------------------
def c4_feas_problem(n=512, d=12, c=2, spread=4.0):
    rng = np.random.default_rng(4)
    X = rng.random((n, d))
    g = ((X[:, 2:] - .5) ** 2).sum(1)
    a, b = .5 * np.pi * X[:, 0], .5 * np.pi * X[:, 1]
    Y = np.column_stack([(1 + g) * np.cos(a) * np.cos(b), (1 + g) * np.cos(a) * np.sin(b), (1 + g) * np.sin(a)])
    G = np.column_stack([X[:, :3].sum(1) - 1.2, 0.4 - X[:, 3] - 0.5 * X[:, 4]])[:, :c] * spread
    models = [ob.GPModel(X, Y[:, i], (0.7 + 0.1 * i) * np.ones(d), 1.0 + i, device=DEV) for i in range(3)]
    models += [ob.GPModel(X, G[:, j], (0.9 + 0.2 * j) * np.ones(d), 1.0, device=DEV) for j in range(c)]
    feasible = np.all(G <= 0, axis=1)
    PF, r = ob.host_prep.calc_pf(Y[feasible]), Y.max(0) + 0.1
    return X, Y, G, models, ob.spec_ehvi_box_feasible(r, PF, c), ob.spec_ehvi_box(r, PF)


@pytest.fixture(scope="module")
def c4():
    return c4_feas_problem()


# ------------------------------------------------------------------------------------------
# 2. reduction to the plain box kind
# ------------------------------------------------------------------------------------------
def test_reduction_to_plain_kind_fp64():
    rng = np.random.default_rng(7)
    for k in (2, 3, 4):
        PF = _sphere(30, k, rng)
        r = PF.max(0) + 0.1
        m = 3001
        mu = PF[rng.integers(0, 30, m)] + rng.normal(0, 0.05, size=(m, k))
        var = (0.05 * rng.uniform(0.5, 1.5, size=(m, k))) ** 2
        plain, bv, bi = _acquire(ob.spec_ehvi_box(r, PF), mu, var)
        for c in (1, 8 - k):
            mu_c = np.full((m, c), -1e3)
            var_c = rng.uniform(0.5, 1.5, size=(m, c))
            feas, fv, fi = _acquire(ob.spec_ehvi_box_feasible(r, PF, c), np.hstack([mu, mu_c]), np.hstack([var, var_c]))
            assert np.array_equal(feas.view(np.int64), plain.view(np.int64)) and (fv, fi) == (bv, bi)


@needs_fast
def test_reduction_to_plain_kind_fast(c4):
    """Constraint models trained on y = -1e3: every PoF is exactly 1.0, in FP32 and FP64, and the fast path's values
    equal the plain kind's bit for bit."""
    X, Y, G, models, spec, plain = c4
    d = X.shape[1]
    deep = [ob.GPModel(X, np.full(len(X), -1e3), (0.9 + 0.2 * j) * np.ones(d), 1.0, device=DEV) for j in range(2)]
    pool = ob.CandidatePool.counter(1 << 14, np.zeros(d), np.ones(d), seed=3)
    for prec in ("fast", "fp64"):
        res = ob.score(models[:3] + deep, spec, pool, precision=prec, want_posterior=True, want_acq=True)
        z = res.mu[3:].cpu().numpy() / np.sqrt(res.var[3:].cpu().numpy() + 1e-5)
        assert z.max() < -10                                 # Phi(-z) rounds to 1.0 in both precisions
        ref = ob.score(models[:3], plain, pool, precision=prec, want_acq=True)
        assert torch.equal(res.acq.view(torch.int64), ref.acq.view(torch.int64))
        assert (res.best_value, res.best_index) == (ref.best_value, ref.best_index)


# ------------------------------------------------------------------------------------------
# 3. the FP32 contract
# ------------------------------------------------------------------------------------------
@needs_fast
def test_fp32_contract(c4):
    X, Y, G, models, spec, plain = c4
    d = X.shape[1]
    pool = ob.CandidatePool.counter(1 << 14, np.zeros(d), np.ones(d), seed=5)
    res = ob.score(models, spec, pool, precision="fast", want_posterior=True, want_acq=True)
    mu, var = res.mu.cpu().numpy().T, res.var.cpu().numpy().T
    v32 = res.acq.cpu().numpy()
    v64, _, _ = _acquire(spec, mu, var)
    e64, _, _ = _acquire(plain, mu[:, :3], var[:, :3])
    pof = _pof64(mu[:, 3:], var[:, 3:], 1e-5)
    np.testing.assert_allclose(v64, e64 * pof, rtol=1e-12, atol=0)
    assert np.all(v32 >= 0) and not np.isnan(v32).any()
    assert np.all(np.abs(v32 - v64) <= 1e-3 * pof * e64.max())
    assert pof.min() < 1e-2 and pof.max() > 0.5


@needs_fast
def test_fp32_deep_infeasible_tail(c4):
    """Constraint posteriors 8 to 12 sigma on the infeasible side (PoF ~1e-15 to 1e-33 per constraint, products far
    below FLT_MIN): the FP32 kernel keeps every value non-zero, within the contract, and selects what FP64 selects."""
    X, Y, G, models, spec, plain = c4
    d = X.shape[1]
    rng = np.random.default_rng(8)
    ones = np.ones(len(X))
    unit = [ob.GPModel(X, ones, (0.9 + 0.2 * j) * np.ones(d), 1.0, device=DEV) for j in range(2)]
    base = ob.CandidatePool.counter(1 << 16, np.zeros(d), np.ones(d), seed=6)
    mu1, var1 = ob.posterior(unit, base, precision="fp64")
    z1 = (mu1 / torch.sqrt(var1 + 1e-5)).cpu().numpy().T         # (m, 2); z of y = s * ones is s * z1
    s = 10.0 / np.median(z1, axis=0)
    zs = z1 * s
    rows = np.flatnonzero(np.all((zs > 8.5) & (zs < 11.5), axis=1))
    assert len(rows) >= 256
    rows = np.sort(rng.choice(rows, min(len(rows), 4096), replace=False))
    pool = ob.CandidatePool.explicit(base.rows(0, base.m, DEV)[torch.as_tensor(rows, device=DEV)])
    cons = [ob.GPModel(X, s[j] * ones, (0.9 + 0.2 * j) * np.ones(d), 1.0, device=DEV) for j in range(2)]
    res = ob.score(models[:3] + cons, spec, pool, precision="fast", want_posterior=True, want_acq=True)
    mu, var = res.mu.cpu().numpy().T, res.var.cpu().numpy().T
    v32 = res.acq.cpu().numpy()
    v64, _, _ = _acquire(spec, mu, var)
    e64, _, _ = _acquire(plain, mu[:, :3], var[:, :3])
    pof = _pof64(mu[:, 3:], var[:, 3:], 1e-5)
    assert pof.max() < 1e-20 and pof.min() > 1e-75
    # non-zero wherever the box sum itself is an FP32 number (a plain FP32 product would flush every value to 0)
    live = e64 > 1e-30
    assert live.mean() > 0.99 and np.all(v32[live] > 0) and np.all(v32 >= 0)
    assert np.all(np.abs(v32 - v64) <= 1e-3 * pof * e64.max())
    _check_selection(v32, v64, res.best_index, rtol=1e-3)


# ------------------------------------------------------------------------------------------
# 4. whole scoring path
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
def test_whole_path(c4, precision):
    X, Y, G, models, spec, plain = c4
    d = X.shape[1]
    pool = ob.CandidatePool.counter(1 << 18, np.zeros(d), np.ones(d), seed=9)
    res = ob.score(models, spec, pool, precision=precision, want_acq=True)
    acq = res.acq.cpu().numpy()
    assert res.best_index == O.argmax_lowest_index(acq) and res.best_value == acq[res.best_index]
    assert acq.max() > 0 and np.all(acq >= 0)
    # reproducible, and only `best` asked for gives the same winner
    again = ob.score(models, spec, pool, precision=precision, want_acq=True)
    assert torch.equal(res.acq.view(torch.int64), again.acq.view(torch.int64))
    only = ob.score(models, spec, pool, precision=precision)
    assert (only.best_value, only.best_index) == (res.best_value, res.best_index)
    # top-k: a stable descending argsort of the same values
    vals, idx = ob.score_topk(models, spec, pool, 257, precision=precision)
    order = np.argsort(-acq, kind="stable")[:257]
    assert np.array_equal(idx, order) and np.array_equal(vals, acq[order])
    # shards of the pool
    shards = [ob.score(models, spec, pool.shard(q, 4), precision=precision) for q in range(4)]
    best = max(shards, key=lambda r: (r.best_value, -r.best_index))
    assert (best.best_value, best.best_index) == (res.best_value, res.best_index)
    assert distributed.score_sharded(models, spec, pool, precision=precision) == (res.best_value, res.best_index)
    # the values are the box sum of the objectives times the feasibility product on the same posteriors
    post = ob.score(models, spec, ob.CandidatePool.counter(4096, np.zeros(d), np.ones(d), seed=9), precision=precision,
                    want_posterior=True, want_acq=True)
    mu, var = post.mu.cpu().numpy().T, post.var.cpu().numpy().T
    e64, _, _ = _acquire(plain, mu[:, :3], var[:, :3])
    pof = _pof64(mu[:, 3:], var[:, 3:], 1e-5)
    tol = 1e-12 if precision == "fp64" else 1e-3
    assert np.all(np.abs(post.acq.cpu().numpy() - e64 * pof) <= tol * pof * e64.max() + 1e-300)


def _best_in_fresh_process(env_extra):
    code = f"""
import json, sys, numpy as np
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, "tests")!r})
import optimobo_b200 as ob
from test_gpu_ehvi_feas import c4_feas_problem
X, Y, G, models, spec, plain = c4_feas_problem()
res = ob.score(models, spec, ob.CandidatePool.counter(1 << 18, np.zeros(12), np.ones(12), seed=9), precision="fast")
print(json.dumps([res.best_value, res.best_index]))
"""
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env_extra), capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return out, tuple(json.loads(out.stdout.strip().splitlines()[-1]))


@needs_fast
def test_never_pruned(c4):
    """The pruned arg-max is for the 2-D EHVI only: a fast, best-only call of this kind never enters it (no
    OMBO_PRUNE_LOG line) and gives what OMBO_NO_PRUNE gives."""
    X, Y, G, models, spec, plain = c4
    mine = ob.score(models, spec, ob.CandidatePool.counter(1 << 18, np.zeros(12), np.ones(12), seed=9),
                    precision="fast")
    logged, a = _best_in_fresh_process({"OMBO_PRUNE_LOG": "1"})
    assert "[prune]" not in logged.stderr
    _, b = _best_in_fresh_process({"OMBO_NO_PRUNE": "1"})
    assert (mine.best_value, mine.best_index) == a == b


# ------------------------------------------------------------------------------------------
# 5. validation
# ------------------------------------------------------------------------------------------
def test_validation():
    rng = np.random.default_rng(1)
    PF = _sphere(10, 3, rng)
    r = PF.max(0) + 0.1
    spec = ob.spec_ehvi_box_feasible(r, PF, 1)
    mu, var = rng.random((64, 9)), rng.random((64, 9)) + 0.1
    _acquire(spec, mu[:, :4], var[:, :4])
    for G in (3, 9):                                             # no constraint model; more models than OMBO_MAX_GP
        with pytest.raises(_cabi.OmboError) as e:
            _acquire(spec, mu[:, :G], var[:, :G])
        assert e.value.code == _cabi.ERR_INVALID
    # through score: three objective GPs and no constraint model
    X = rng.random((32, 2))
    models = [ob.GPModel(X, X[:, 0] + i, np.ones(2), 1.0, device=DEV) for i in range(3)]
    bare = ob.AcquisitionSpec(kind=_cabi.ACQ_EHVI_BOX_FEAS, n_obj=3, ref=tuple(r), stripes=spec.stripes,
                              cells=spec.cells, var_eps=spec.var_eps, n_models=3)
    with pytest.raises(_cabi.OmboError) as e:
        ob.score(models, bare, ob.CandidatePool.counter(64, np.zeros(2), np.ones(2)))
    assert e.value.code == _cabi.ERR_INVALID


# ------------------------------------------------------------------------------------------
# 6. batches
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
def test_batch_matches_brute_force_believer(precision):
    X, Y, G, models, spec0, plain = c4_feas_problem(n=256, d=8)
    r = np.asarray(spec0.ref)
    feasible = np.all(G <= 0, axis=1)
    PF = ob.host_prep.calc_pf(Y[feasible])

    def spec_for(Yb):
        Yb = np.asarray(Yb).reshape(-1, 5)
        ok = Yb[np.all(Yb[:, 3:] <= 0, axis=1) & np.all(Yb[:, :3] <= r, axis=1), :3]
        return ob.spec_ehvi_box_feasible(r, ob.host_prep.calc_pf(np.vstack([PF, ok])) if len(ok) else PF, 2)

    pool = ob.CandidatePool.counter(1 << 16, np.zeros(8), np.ones(8), seed=11)
    q = 4
    Xq, neg, idx, cert = ob.propose_batch(models, spec_for, pool, q, precision=precision)
    assert Xq.shape == (q, 8) and len(set(idx.tolist())) == q and not cert.any()
    want, gaps, scales = brute_force(models, spec_for, pool, q, precision)
    same_selection(list(idx), want, gaps, scales, 2e-3 if precision == "fast" else 2e-6)


# ------------------------------------------------------------------------------------------
# 7. the constrained optimiser on BNH
# ------------------------------------------------------------------------------------------
class BNH(Problem):                      # README example 2
    def __init__(self):
        super().__init__(n_var=2, n_obj=2, n_ieq_constr=2, vtype=float)
        self.xl = np.zeros(self.n_var)
        self.xu = np.array([5.0, 3.0])

    def _evaluate(self, x, out, *args, **kwargs):
        out["F"] = [4 * x[:, 0] ** 2 + 4 * x[:, 1] ** 2, (x[:, 0] - 5) ** 2 + (x[:, 1] - 5) ** 2]

    def _evaluate_constraints(self, x, out, *args, **kwargs):
        out["G"] = [(1 / 25) * ((x[:, 0] - 5) ** 2 + x[:, 1] ** 2 - 25),
                    -1 / 7.7 * ((x[:, 0] - 8) ** 2 + (x[:, 1] + 3) ** 2 - 7.7)]


KW = dict(n_candidates=1 << 14, seed=0, device=DEV, max_f_eval=200)


class _Recording(MultiSurrogateOptimiser):
    def _propose(self, models, spec):
        self.kinds = getattr(self, "kinds", []) + [(spec.kind, len(models))]
        return super()._propose(models, spec)


@pytest.mark.parametrize("batch_size", [1, 2])
def test_optimiser_bnh(batch_size):
    opt = _Recording(BNH(), [0, 0], [140, 50], ehvi="box", constrained=True, batch_size=batch_size, **KW)
    res = opt.solve(budget=5, n_init_samples=10)
    assert isinstance(res, result.Constrained_Res)
    assert res.ysample.shape == (15, 2) and res.Xsample.shape == (15, 2) and res.gsample.shape == (15, 2)
    np.testing.assert_allclose(res.gsample, BNH().evaluate_constraints(res.Xsample))
    np.testing.assert_allclose(res.ysample, BNH().evaluate(res.Xsample))
    feasible = np.all(res.gsample <= 0, axis=1)
    assert len(res.y_feasible) == feasible.sum() and len(res.y_feasible) + len(res.y_infeasible) == 15
    assert len(res.pf_approx) >= 1 and res.pf_inputs.shape == (len(res.pf_approx), 2)
    assert np.all(BNH().evaluate_constraints(res.pf_inputs) <= 0)
    assert ob.host_prep.pareto_mask(res.pf_approx).all()
    hv = res.hypervolume_convergence
    assert len(hv) == (5 if batch_size == 1 else 3)
    assert all(b >= a for a, b in zip(hv, hv[1:]))
    assert hv[0] == ob.host_prep.hypervolume(res.ysample[:10][feasible[:10]], [140, 50])
    if batch_size == 1:
        assert opt.kinds == [(_cabi.ACQ_EHVI_BOX_FEAS, 4)] * 5
    else:
        assert [t["batch"] for t in res.timings] == [2, 2, 1] and sum(t["certified"] for t in res.timings) == 0


def test_optimiser_unconstrained_default_unchanged():
    kw = dict(KW, hyperparameters=(np.ones(2), 1.0))
    a = MultiSurrogateOptimiser(BNH(), [0, 0], [140, 50], ehvi="box", **kw).solve(budget=3, n_init_samples=8)
    b = MultiSurrogateOptimiser(BNH(), [0, 0], [140, 50], ehvi="box", constrained=False, **kw).solve(budget=3,
                                                                                                   n_init_samples=8)
    assert type(a) is type(b) is result.Res
    np.testing.assert_array_equal(a.ysample, b.ysample)
    np.testing.assert_array_equal(a.Xsample, b.Xsample)
    assert a.hypervolume_convergence == b.hypervolume_convergence
