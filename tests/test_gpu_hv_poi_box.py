"""GPU: the hypervolume-based probability of improvement for 2 to 4 objectives over the box decomposition
(OMBO_ACQ_HV_POI_BOX, k_acquire_box in its HV-PoI mode) against the grid oracle and a 50-digit value in the tails,
against the 2-D cell kind OMBO_ACQ_HV_POI, in both precisions, through every scoring entry and EMO."""
import mpmath as mp
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi, distributed  # noqa: E402
from optimobo_b200.algorithms import EMO  # noqa: E402
from optimobo_b200.problem import Problem  # noqa: E402
from oracle import oracle as O  # noqa: E402
from hv_poi_oracle import hv_poi_box_batched, hv_poi_grid_batched, region_ref  # noqa: E402
from test_gpu_ehvi_box import _c4  # noqa: E402
from test_gpu_parity import _check_selection  # noqa: E402

DEV = "cuda:0"
needs_fast = pytest.mark.skipif(not _cabi.fast_path_available(), reason="fast path not built")


def _sphere(P, k, rng):
    X = np.abs(rng.normal(size=(P, k)))
    return X / np.linalg.norm(X, axis=1, keepdims=True)


def _posteriors(PF, m, rng, spread=0.05, sd=0.05):
    k = PF.shape[1]
    mu = PF[rng.integers(0, len(PF), m)] + rng.normal(0, spread, size=(m, k))
    var = (sd * rng.uniform(0.5, 1.5, size=(m, k))) ** 2
    return mu, var


def _acquire(spec, mu, var, index_base=0):
    acq, bv, bi = ob.acquire_from_posterior(spec, mu.T, var.T, DEV, index_base=index_base)
    return acq.cpu().numpy(), bv, bi


def _hv_poi_mp(spec, mu, var):
    """PoI * Imp over the spec's own (clamped) boxes in 50 digits.  A box's mass is taken as a difference of two
    upper tails above the mean, so the value is exact where every box lies far above it."""
    mp.mp.dps = 50
    table, boxes = np.asarray(spec.stripes), np.asarray(spec.cells).astype(np.int64)
    k = table.shape[0]
    out = []
    for mr, vr in zip(mu, var):
        m_ = [mp.mpf(x) for x in mr]
        s_ = [mp.sqrt(mp.mpf(x) + mp.mpf(1e-5)) for x in vr]
        poi = imp = mp.mpf(0)
        for bx in boxes:
            p = e = mp.mpf(1)
            for i in range(k):
                u, l = mp.mpf(table[i, bx[0, i]]), mp.mpf(table[i, bx[1, i]])
                zl, zu = (l - m_[i]) / s_[i], (u - m_[i]) / s_[i]
                p *= mp.ncdf(-zl) - mp.ncdf(-zu)
                e *= max(u - max(l, m_[i]), mp.mpf(0))
            poi += p
            imp += e
        out.append(float(poi * imp))
    return np.array(out)


# ------------------------------------------------------------------------------------------
# K4 alone
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,P", [(2, 40), (3, 40), (4, 12)])
@pytest.mark.parametrize("maxp_side", ["above", "below"])
def test_fp64_vs_grid_oracle_and_tails(k, P, maxp_side):
    rng = np.random.default_rng(k * 100 + P + (maxp_side == "below"))
    PF = _sphere(P, k, rng)
    ideal = PF.min(0) - 0.05
    maxp = PF.max(0) + (0.1 if maxp_side == "above" else -0.1)
    spec = ob.spec_hv_poi_box(ideal, maxp, PF)
    r = region_ref(PF, maxp)
    mu, var = _posteriors(PF, 2000, rng)
    # 10 to 30 sigma below the ideal point in objective 0 (10 to 11 in the others, so that the value stays a normal
    # double for k = 4): every box lies above the mean
    sd = np.sqrt(var[:10] + 1e-5)
    z = np.column_stack([rng.uniform(10, 30, 10)] + [rng.uniform(10, 11, 10)] * (k - 1))
    mu[:10] = ideal - z * sd
    mu[10:20] = PF[rng.integers(0, P, 10)]
    mu[10:20, 0] = r[0] + rng.uniform(1e-3, 1.0, 10)               # beyond r' in one objective: exactly 0
    got, bv, bi = _acquire(spec, mu, var)
    want = hv_poi_grid_batched(mu, var, PF, ideal, maxp)
    np.testing.assert_allclose(got[20:], want[20:], rtol=1e-9, atol=1e-14 * np.abs(want).max())
    assert np.all(got[10:20] == 0)
    tail = _hv_poi_mp(spec, mu[:10], var[:10])
    assert np.all(tail > 1e-300)
    np.testing.assert_allclose(got[:10], tail, rtol=1e-9)
    np.testing.assert_allclose(want[:10], tail, rtol=1e-9)
    assert bi == O.argmax_lowest_index(got) and bv == got[bi]


def test_nan_ranks_as_minus_inf():
    rng = np.random.default_rng(2)
    PF = _sphere(20, 3, rng)
    spec = ob.spec_hv_poi_box(PF.min(0), PF.max(0) + 0.1, PF)
    mu, var = _posteriors(PF, 300, rng)
    mu[5, 1] = np.nan
    var[7, 2] = np.nan
    got, bv, bi = _acquire(spec, mu, var)
    assert np.isnan(got[5]) and np.isnan(got[7]) and bi == O.argmax_lowest_index(got) and bv == got[bi]


def test_k2_equals_the_cell_kind(golden):
    """Ideal point at or below the front: the box kind on decompose_into_cells' region equals OMBO_ACQ_HV_POI.  That
    kind subtracts two Phi near 1 for a cell above the mean (~1e-16 absolute), hence the absolute floor."""
    cases = [(golden["acq_out_calc_pf"], golden["emo_in_ideal"], golden["emo_in_max"], golden["acq_in_mu2"],
              golden["acq_in_var2"])]
    rng = np.random.default_rng(12)
    for side in (0.15, -0.15):
        Y = rng.random((40, 2))
        PF = ob.host_prep.calc_pf(Y)
        mu, var = _posteriors(PF, 3000, rng, spread=0.2)
        cases.append((PF, Y.min(0) - np.array([0.0, 0.05]), Y.max(0) + side, mu, var))
    for PF, ideal, maxp, mu, var in cases:
        assert np.all(PF >= ideal)
        box, bv, bi = _acquire(ob.spec_hv_poi_box(ideal, maxp, PF), mu, var)
        cells, cv, ci = _acquire(ob.spec_hv_poi(ob.host_prep.decompose_into_cells(PF, ideal, maxp)), mu, var)
        np.testing.assert_allclose(box, cells, rtol=1e-12, atol=1e-16)
        assert box.max() > 0


@pytest.mark.parametrize("m", [1, 255, 257, 5001])
def test_ragged_m_index_base_and_reproducibility(m):
    rng = np.random.default_rng(m)
    PF = _sphere(50, 3, rng)
    ideal, maxp = PF.min(0), PF.max(0) + 0.1
    mu, var = _posteriors(PF, m, rng)
    spec = ob.spec_hv_poi_box(ideal, maxp, PF)
    base = 10 ** 9 + 17
    got, bv, bi = _acquire(spec, mu, var, index_base=base)
    want = hv_poi_box_batched(mu, var, PF, ideal, maxp)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-14 * max(np.abs(want).max(), 1e-300))
    assert bi == base + O.argmax_lowest_index(got) and bv == got[bi - base]
    again, bv2, bi2 = _acquire(spec, mu, var, index_base=base)
    assert np.array_equal(got.view(np.int64), again.view(np.int64)) and (bv2, bi2) == (bv, bi)


@needs_fast
@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_fp32_kernel(offset):
    """The FP32 K4 of the fast mode on the fast path's own posteriors.  offset = 1e3 moves the training targets and
    the front together, so t - mu ~ 1 must keep its digits next to t, mu ~ 1e3."""
    X, Y, ells, sf2 = _c4(n=256, d=6)
    models = [ob.GPModel(X, Y[:, i] + offset, ells[i], sf2[i], device=DEV) for i in range(3)]
    PF = ob.host_prep.calc_pf(Y) + offset
    ideal, maxp = PF.min(0), PF.max(0) + 0.1
    spec = ob.spec_hv_poi_box(ideal, maxp, PF)
    pool = ob.CandidatePool.counter(1 << 12, np.zeros(6), np.ones(6), seed=5)
    res = ob.score(models, spec, pool, precision="fast", want_posterior=True, want_acq=True)
    mu, var = res.mu.cpu().numpy().T, res.var.cpu().numpy().T
    got = res.acq.cpu().numpy()
    want = hv_poi_grid_batched(mu, var, PF, ideal, maxp)
    assert want.max() > 0
    np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-3 * np.abs(want).max())
    f64, _, _ = _acquire(spec, mu, var)
    np.testing.assert_allclose(f64, want, rtol=1e-9, atol=1e-12 * np.abs(want).max())
    big = np.abs(f64) > 1e-3 * np.abs(f64).max()
    assert big.sum() >= 50
    print(f"offset {offset}: FP32 vs FP64 kernel, max relative difference above 1e-3 max: "
          f"{np.max(np.abs(got[big] / f64[big] - 1)):.3e} over {big.sum()} values")
    np.testing.assert_allclose(got[big], f64[big], rtol=1e-4)


# ------------------------------------------------------------------------------------------
# whole path at the C4 shape: DTLZ2, n = 512, d = 12, k = 3
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c4():
    X, Y, ells, sf2 = _c4()
    models = [ob.GPModel(X, Y[:, i], ells[i], sf2[i], device=DEV) for i in range(3)]
    PF, ideal, maxp = ob.host_prep.calc_pf(Y), Y.min(0), Y.max(0)
    return X, Y, ells, sf2, models, ob.spec_hv_poi_box(ideal, maxp, PF), PF, ideal, maxp


@pytest.mark.parametrize("precision", ["fp64", pytest.param("fast", marks=needs_fast)])
def test_full_path_c4(c4, precision):
    X, Y, ells, sf2, models, spec, PF, ideal, maxp = c4
    m, d = 1 << 12, X.shape[1]
    lo, hi = np.zeros(d), np.ones(d)
    pool = ob.CandidatePool.counter(m, lo, hi, seed=2)
    Xc = O.candidates_from_counter(2, 0, m, lo, hi)
    post = [O.gp_posterior(O.gp_fit_state(X, Y[:, i], ells[i], sf2[i]), Xc) for i in range(3)]
    mu_o, var_o = np.array([p[0] for p in post]).T, np.array([p[1] for p in post]).T
    want = hv_poi_box_batched(mu_o, var_o, PF, ideal, maxp)
    res = ob.score(models, spec, pool, precision=precision, want_acq=True)
    got = res.acq.cpu().numpy()
    tol = 1e-5 if precision == "fp64" else 2e-3
    np.testing.assert_allclose(got, want, rtol=tol, atol=tol * np.abs(want).max())
    _check_selection(got, want, res.best_index, rtol=1e-6 if precision == "fp64" else 1e-3)
    x, neg, idx = ob.propose(models, spec, pool, precision=precision)
    assert idx == res.best_index and np.array_equal(x, Xc[idx]) and neg == -res.best_value


@pytest.mark.parametrize("precision", ["fp64", pytest.param("fast", marks=needs_fast)])
def test_spec_on_device_equals_host(c4, precision):
    X, Y, ells, sf2, models, spec, PF, ideal, maxp = c4
    dspec = ob.spec_hv_poi_box(ideal, maxp, PF, device=DEV)
    assert torch.is_tensor(dspec.stripes) and dspec.stripes.is_cuda
    assert np.array_equal(dspec.stripes.cpu().numpy(), spec.stripes)
    assert np.array_equal(dspec.cells.cpu().numpy(), spec.cells)
    pool = ob.CandidatePool.counter(1 << 16, np.zeros(12), np.ones(12), seed=4)
    a = ob.score(models, spec, pool, precision=precision, want_acq=True)
    b = ob.score(models, dspec, pool, precision=precision, want_acq=True)
    assert torch.equal(a.acq.view(torch.int64), b.acq.view(torch.int64))
    assert (a.best_value, a.best_index) == (b.best_value, b.best_index)


def test_other_entry_points(c4):
    """score_topk, distributed.score_sharded, propose and polish take the kind."""
    X, Y, ells, sf2, models, spec, PF, ideal, maxp = c4
    d = X.shape[1]
    pool = ob.CandidatePool.counter(1 << 18, np.zeros(d), np.ones(d), seed=9)
    whole = ob.score(models, spec, pool, want_acq=True)
    acq = whole.acq.cpu().numpy()
    vals, idx = ob.score_topk(models, spec, pool, 257)
    order = np.argsort(-acq, kind="stable")[:257]
    assert np.array_equal(idx, order) and np.array_equal(vals, acq[order])
    assert distributed.score_sharded(models, spec, pool) == (whole.best_value, whole.best_index)
    rows, tv = ob.top_candidates(models, spec, pool, 4, head=1 << 14)
    np.testing.assert_allclose(ob.evaluate(models, spec, rows), tv, rtol=1e-9)
    xp, vp, per = ob.polish(models, spec, rows[:2], np.zeros(d), np.ones(d), max_iter=5)
    assert vp >= tv[0] * (1 - 1e-9) and per.shape == (2,)
    x, neg, _ = ob.propose(models, spec, pool, refine_rounds=1, refine_candidates=1 << 12)
    assert -neg >= whole.best_value and x.shape == (d,)
    np.testing.assert_allclose(ob.hypervolume_based_PoI_box(x, models, ideal, maxp, PF), [-neg], rtol=1e-9)


# ------------------------------------------------------------------------------------------
# size limits
# ------------------------------------------------------------------------------------------
def test_largest_front_scores_and_one_more_raises():
    rng = np.random.default_rng(3)
    P = _cabi.EHVI_BOX_MAX_BREAKS - 2
    F = ob.host_prep.calc_pf(_sphere(4 * P, 3, rng))[:P]
    assert len(F) == P
    ideal, maxp = F.min(0), F.max(0) + 0.1
    spec = ob.spec_hv_poi_box(ideal, maxp, F)
    assert spec.stripes.shape[1] == _cabi.EHVI_BOX_MAX_BREAKS
    mu, var = _posteriors(F, 2000, rng)
    got, _, _ = _acquire(spec, mu, var)
    want = hv_poi_box_batched(mu[:64], var[:64], F, ideal, maxp)
    np.testing.assert_allclose(got[:64], want, rtol=1e-9, atol=1e-14 * np.abs(want).max())
    G = ob.host_prep.calc_pf(_sphere(4 * (P + 1), 3, np.random.default_rng(4)))[:P + 1]
    with pytest.raises(_cabi.OmboError, match="breakpoints"):
        _acquire(ob.spec_hv_poi_box(G.min(0), G.max(0) + 0.1, G), mu, var)


# ------------------------------------------------------------------------------------------
# EMO for 3 and 4 objectives
# ------------------------------------------------------------------------------------------
class DTLZ2(Problem):
    def __init__(self, n_var=6, n_obj=3):
        super().__init__(n_var=n_var, n_obj=n_obj, xl=np.zeros(n_var), xu=np.ones(n_var))

    def _evaluate(self, x, out, *args, **kwargs):
        k = self.n_obj
        g = ((x[:, k - 1:] - 0.5) ** 2).sum(1)
        th = 0.5 * np.pi * x[:, :k - 1]
        F = []
        for i in range(k):
            f = 1 + g
            for j in range(k - 1 - i):
                f = f * np.cos(th[:, j])
            if i > 0:
                f = f * np.sin(th[:, k - 1 - i])
            F.append(f)
        out["F"] = F


class _Recording(EMO):
    def _propose(self, models, spec):
        x, neg = super()._propose(models, spec)
        self.seen = getattr(self, "seen", []) + [(spec.kind, -neg)]
        return x, neg


@pytest.mark.parametrize("n_obj", [3, 4])
def test_emo_solve(n_obj):
    opt = _Recording(DTLZ2(n_obj=n_obj), np.zeros(n_obj), np.full(n_obj, 2.5), n_candidates=1 << 14, seed=0,
                     device=DEV, max_f_eval=200)
    res = opt.solve(budget=3, n_init_samples=12)
    assert res.ysample.shape == (15, n_obj) and np.all(np.isfinite(res.ysample))
    assert [kind for kind, _ in opt.seen] == [_cabi.ACQ_HV_POI_BOX] * 3
    assert max(v for _, v in opt.seen) > 0
