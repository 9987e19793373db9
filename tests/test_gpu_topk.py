"""GPU: the exact top-k of ombo_score_topk equals a stable descending argsort (NaN as -inf, ties to the lowest index)
of the values ombo_score writes to out_acq, bit for bit: every acquisition path (fused f8c 2-D EHVI in both
semantics, k_acquire, k_acquire_box), both precisions, counter / f64 / f32 pools, ragged sizes and m < k, a non-zero
index base, duplicated rows, an all-zero pool (millions-way ties are the same logic as these thousands) and several
passes per call (OMBO_CHUNK_LOG2=10 in a fresh process).  k = 1 is ombo_score's arg-max, pruned path included."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi  # noqa: E402
from oracle import oracle as O  # noqa: E402

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
D = 10


def problem(n=1024):
    """C5-like: ZDT1 (plus a third objective for the box EHVI) on n points in 10-D, injected hyper-parameters."""
    rng = np.random.default_rng(0)
    X = rng.random((n, D))
    f1 = X[:, 0]
    g = 1 + 9.0 / (D - 1) * X[:, 1:].sum(1)
    Y = np.column_stack([f1, g * (1 - np.sqrt(f1 / g)), g * (1 - X[:, 1]) + 0.5 * f1])
    models = [ob.GPModel(X, Y[:, i], [0.7, 0.8, 0.9][i] * np.ones(D), [1.0, 2.0, 1.5][i], device=DEV)
              for i in range(3)]
    return models, Y


@pytest.fixture(scope="module")
def setup():
    models, Y = problem()
    cache = ob.host_prep.cached_samples(2, 5, seed=0)
    PF, r = ob.host_prep.calc_pf(Y[:, :2]), Y[:, :2].max(0)
    PF3, r3 = ob.host_prep.calc_pf(Y), Y.max(0)
    specs = {
        "ehvi_ref": (models[:2], ob.spec_ehvi(r, PF, cache, "reference")),
        "ehvi_exact": (models[:2], ob.spec_ehvi(r, PF, cache, "exact")),
        "ei": (models[:1], ob.spec_ei(float(Y[:, 0].min()))),
        "box3": (models, ob.spec_ehvi_box(r3, PF3)),
        "hv_poi": (models[:2], ob.spec_hv_poi(O.decompose_into_cells_2d(PF, Y[:, :2].min(0), r))),
        "cei": (models[:2], ob.spec_constrained_ei(float(Y[:, 0].min()), 1)),
    }
    return models, specs, (PF, r, cache)


def reference_topk(acq, k, base):
    a = np.where(np.isnan(acq), -np.inf, acq)
    order = np.argsort(-a, kind="stable")[:k]
    vals = np.full(k, -np.inf)
    idx = np.full(k, -1, dtype=np.int64)
    vals[:len(order)] = a[order]
    idx[:len(order)] = order + base
    return vals, idx


def check(models, spec, pool, k, precision):
    acq = ob.score(models, spec, pool, precision=precision, want_acq=True, want_best=False).acq.cpu().numpy()
    vals, idx = ob.score_topk(models, spec, pool, k, precision=precision)
    want_v, want_i = reference_topk(acq, k, pool.index_base)
    np.testing.assert_array_equal(idx, want_i)
    np.testing.assert_array_equal(vals, want_v)          # -0 ranks and is reported as +0: equal as values
    return vals, idx


def pools(m):
    counter = ob.CandidatePool.counter(m, np.zeros(D), np.ones(D), seed=m)
    rows = counter.rows(0, m, DEV)
    return {"counter": counter, "f64": ob.CandidatePool.explicit(rows),
            "f32": ob.CandidatePool.explicit(rows.to(torch.float32))}


@pytest.mark.parametrize("kind", ["ehvi_ref", "ehvi_exact", "ei", "box3", "hv_poi", "cei"])
@pytest.mark.parametrize("precision", ["fp64", "fast"])
def test_topk_matches_stable_argsort(setup, kind, precision):
    if precision == "fast" and not _cabi.fast_path_available():
        pytest.skip("fast path not built")
    _, specs, _ = setup
    models, spec = specs[kind]
    for m in (1, 63, 5001, 70001):
        for name, pool in pools(m).items():
            for k in (1, 100, 4096):
                check(models, spec, pool, k, precision)


def test_index_base_duplicates_and_k_max(setup):
    _, specs, _ = setup
    models, spec = specs["ehvi_exact"]
    prec = "fast" if _cabi.fast_path_available() else "fp64"
    pool = ob.CandidatePool.counter(3 << 16, np.zeros(D), np.ones(D), seed=9, index_base=(1 << 33) + 7)
    check(models, spec, pool, 4096, prec)
    check(models, spec, pool, _cabi.TOPK_MAX, prec)
    base = ob.CandidatePool.counter(1 << 14, np.zeros(D), np.ones(D), seed=4)
    _, idx = ob.score_topk(models, spec, base, 3, precision=prec)
    rows = base.rows(0, 1 << 14, DEV)
    w = int(idx[0])
    X = torch.cat([rows, rows[w:w + 1].repeat(5, 1), rows], 0)          # the winner at seven indices
    for dtype in (torch.float64, torch.float32):
        vals, idx = check(models, spec, ob.CandidatePool.explicit(X.to(dtype)), 64, prec)
        if dtype == torch.float64:
            assert list(idx[:7]) == [w] + list(range(1 << 14, (1 << 14) + 5)) + [(1 << 14) + 5 + w]
            assert len(set(vals[:7].tolist())) == 1


def test_all_zero_pool_ties_to_lowest_indices(setup):
    models, _, (PF, r, cache) = setup
    far = ob.spec_ehvi(r, PF - 50.0, cache, "exact")      # every value underflows to 0
    for prec in ("fp64", "fast") if _cabi.fast_path_available() else ("fp64",):
        pool = ob.CandidatePool.counter(70001, np.zeros(D), np.ones(D), seed=2)
        vals, idx = check(models[:2], far, pool, 4096, prec)
        assert np.all(vals == 0.0) and list(idx) == list(range(4096))


def test_k1_is_the_argmax_pruned_path_included(setup):
    _, specs, _ = setup
    for kind in ("ehvi_exact", "ehvi_ref", "ei", "box3"):
        models, spec = specs[kind]
        for prec in ("fp64", "fast") if _cabi.fast_path_available() else ("fp64",):
            for m, seed in ((1 << 16, 1), (70001, 5), (1 << 20, 3)):
                pool = ob.CandidatePool.counter(m, np.zeros(D), np.ones(D), seed=seed)
                res = ob.score(models, spec, pool, precision=prec)          # fast exact EHVI: the pruned path
                vals, idx = ob.score_topk(models, spec, pool, 1, precision=prec)
                assert (float(vals[0]), int(idx[0])) == (res.best_value, res.best_index), (kind, prec, m)


def test_top_candidates_whole_pool(setup):
    _, specs, _ = setup
    models, spec = specs["ehvi_exact"]
    pool = ob.CandidatePool.counter(300001, np.zeros(D), np.ones(D), seed=7)
    X, vals = ob.top_candidates(models, spec, pool, 16, head=None)
    v, idx = ob.score_topk(models, spec, pool, 16)
    np.testing.assert_array_equal(vals, v)
    np.testing.assert_array_equal(X, pool.rows(0, pool.m, DEV).cpu().numpy()[idx])
    Xh, vh = ob.top_candidates(models, spec, pool, 16)
    vh_ref, _ = ob.score_topk(models, spec, ob.CandidatePool.counter(1 << 18, np.zeros(D), np.ones(D), seed=7), 16)
    np.testing.assert_array_equal(vh, vh_ref)


MULTI_PASS = r"""
import json, sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import optimobo_b200 as ob
from test_gpu_topk import problem, pools, reference_topk, D
models, Y = problem()
cache = ob.host_prep.cached_samples(2, 5, seed=0)
PF, r = ob.host_prep.calc_pf(Y[:, :2]), Y[:, :2].max(0)
specs = [(models[:2], ob.spec_ehvi(r, PF, cache, "exact")), (models[:2], ob.spec_ehvi(r, PF, cache, "reference")),
         (models[:1], ob.spec_ei(float(Y[:, 0].min()))), (models, ob.spec_ehvi_box(Y.max(0), ob.host_prep.calc_pf(Y))),
         (models[:2], ob.spec_ehvi(r, PF - 50.0, cache, "exact"))]
bad = 0
for prec in ("fp64", "fast"):
    for models_, spec in specs:
        for m in (5001, 70001):
            for pool in pools(m).values():
                acq = ob.score(models_, spec, pool, precision=prec, want_acq=True, want_best=False).acq.cpu().numpy()
                for k in (1, 700, 4096):
                    v, i = ob.score_topk(models_, spec, pool, k, precision=prec)
                    wv, wi = reference_topk(acq, k, pool.index_base)
                    bad += int(not (np.array_equal(v, wv) and np.array_equal(i, wi)))
print(json.dumps(bad))
"""


def test_several_passes_per_call():
    code = MULTI_PASS.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, OMBO_CHUNK_LOG2="10"), capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1]) == 0
