"""GPU: stage 1 of the pruned arg-max (the mean-only bound, posterior_mean8.cu) and the two-stage cascade in ombo_score.

(a) The stage-1 launch gives both GPs' means bit for bit as the full f8c launch (n_pad 256 / 384 / 768 / 1024, d 1..12,
    Matern and RBF, counter / f32 / f64 pools, ragged m), and its bound is >= the full value of every candidate up to
    the FP32 contract.
(b) The cascade returns the unpruned call's (value, index) and the depth-1-only call's (OMBO_PRUNE_STAGE1=0) over pool
    sizes, index bases and shards, duplicated rows, an all-zero pool and a forced-small cap at each stage."""
import ctypes as C
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

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cabi.fast_path_available(), reason="fast path not built")]


def problem(n=1024, d=10, kernels=("matern52", "matern52"), noise=0.0):
    """bench.py's C5 workload shape (ZDT1, injected hyper-parameters) at any n, d and kernel pair; noise is the
    noise variance as a share of each GP's signal variance."""
    rng = np.random.default_rng(0)
    X = rng.random((n, d))
    f1 = X[:, 0]
    g = 1 + 9.0 / max(d - 1, 1) * X[:, 1:].sum(1)
    Y = np.column_stack([f1, g * (1 - np.sqrt(f1 / g))])
    sf2 = [1.0, 2.0]
    models = [ob.GPModel(X, Y[:, i], [0.7, 0.8][i] * np.ones(d), sf2[i], noise=noise * sf2[i], kernel=kernels[i],
                         device=DEV) for i in range(2)]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    spec = ob.spec_ehvi(r, PF, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
    return models, spec, PF, r


def stage1(models, spec, pool):
    """mu [2, m], UB [m] and the largest bound of the stage-1 launch, through the library's test hook."""
    lib = _cabi.lib()
    fn = lib.ombo_debug_mean8
    fn.argtypes = [C.c_void_p, C.POINTER(_cabi.Gp), C.POINTER(_cabi.Pool), C.POINTER(_cabi.Acq), C.c_void_p,
                   C.c_void_p, C.c_void_p, C.c_void_p]
    mu = torch.empty((2, pool.m), dtype=torch.float64, device=DEV)
    ub = torch.empty(pool.m, dtype=torch.float64, device=DEV)
    best = torch.empty(2, dtype=torch.int64, device=DEV)
    gps = (_cabi.Gp * 2)(*[m.c_struct(1e-15) for m in models])
    p, a = pool.c_struct(), spec.c_struct(torch.device(DEV))
    ctx = _cabi.Context.get(0)
    _cabi.check(fn(ctx.handle, gps, C.byref(p), C.byref(a), C.c_void_p(mu.data_ptr()), C.c_void_p(ub.data_ptr()),
                   C.c_void_p(best.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return mu, ub, best


def pools(d, m):
    cnt = ob.CandidatePool.counter(m, np.zeros(d), np.ones(d), seed=3)
    rows = cnt.rows(0, m, DEV)
    return [cnt, ob.CandidatePool.explicit(rows.to(torch.float32)), ob.CandidatePool.explicit(rows + 1e-3)]


@pytest.mark.parametrize("n", [256, 300, 700, 1024])          # n_pad 256, 384, 768, 1024
def test_stage1_mean_is_exact_n_pad(n):
    models, spec, _, _ = problem(n)
    assert all(m.plane_format == "f8c" for m in models)
    for pool in pools(10, 70001):
        full = ob.score(models, spec, pool, precision="fast", want_posterior=True, want_acq=True)
        mu, ub, _ = stage1(models, spec, pool)
        assert torch.equal(mu, full.mu), (n, pool.m)
        # the bound: never below the full value beyond the FP32 contract of the acquisition
        assert bool((ub >= full.acq - 2e-3 * float(ub.max())).all())


@pytest.mark.parametrize("d", list(range(1, 13)))
@pytest.mark.parametrize("kernels", [("matern52", "matern52"), ("rbf", "rbf"), ("matern52", "rbf"), ("rbf", "matern52")])
def test_stage1_mean_is_exact_d_kernel(d, kernels):
    # noise 2 % of sigma_f2 keeps (max L_ii / min L_ii)^2 near 50 at every d, under the f8c format's limit of 100: 300
    # noise-free points at small d are far too ill-conditioned for it
    models, spec, _, _ = problem(300, d, kernels, noise=2e-2)
    assert all(m.plane_format == "f8c" for m in models), (d, kernels)
    for pool in pools(d, 4099):
        full = ob.score(models, spec, pool, precision="fast", want_posterior=True)
        mu, _, _ = stage1(models, spec, pool)
        assert torch.equal(mu, full.mu), (d, kernels)


def test_stage1_largest_bound():
    models, spec, _, _ = problem()
    pool = ob.CandidatePool.counter(100003, np.zeros(10), np.ones(10), seed=5, index_base=1 << 33)
    _, ub, best = stage1(models, spec, pool)
    w = torch.where(torch.isnan(ub), torch.full_like(ub, -np.inf), ub)
    assert best[:1].view(torch.float64).item() == float(w.max())
    assert int(best[1]) == (1 << 33) + int(torch.nonzero(w == w.max())[0])


@pytest.fixture(scope="module")
def c5():
    return problem()


def pruned(models, spec, pool):
    res = ob.score(models, spec, pool, precision="fast")
    return res.best_value, res.best_index


def unpruned(models, spec, pool):
    res = ob.score(models, spec, pool, precision="fast", want_acq=True)          # out_acq: not eligible
    return res.best_value, res.best_index


@pytest.mark.parametrize("m", [1, 63, 257, (1 << 20) + 5, 1 << 24])
def test_cascade_parity_sizes(c5, m):
    models, spec, _, _ = c5
    for seed in ((1, 2) if m < (1 << 24) else (1,)):
        pool = ob.CandidatePool.counter(m, np.zeros(10), np.ones(10), seed=seed)
        assert pruned(models, spec, pool) == unpruned(models, spec, pool), (m, seed)


def test_cascade_index_base_and_shards(c5):
    models, spec, _, _ = c5
    pool = ob.CandidatePool.counter(3 << 18, np.zeros(10), np.ones(10), seed=9, index_base=(1 << 33) + 7)
    assert pruned(models, spec, pool) == unpruned(models, spec, pool)
    for rank in range(3):
        shard = pool.shard(rank, 3)
        assert pruned(models, spec, shard) == unpruned(models, spec, shard)


def test_cascade_duplicates_tie_to_lowest_index(c5):
    models, spec, _, _ = c5
    base = ob.CandidatePool.counter(1 << 16, np.zeros(10), np.ones(10), seed=4)
    _, i_best = unpruned(models, spec, base)
    rows = base.rows(0, 1 << 16, DEV)
    X = torch.cat([rows, rows[i_best:i_best + 1].repeat(5, 1), rows], 0)
    for dtype in (torch.float64, torch.float32):
        pool = ob.CandidatePool.explicit(X.to(dtype))
        v, i = pruned(models, spec, pool)
        assert (v, i) == unpruned(models, spec, pool)
        if dtype == torch.float64:
            assert i == i_best


def test_cascade_all_zero_pool(c5):
    models, spec, PF, r = c5
    far = ob.spec_ehvi(r, PF - 50.0, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
    pool = ob.CandidatePool.counter(4096, np.zeros(10), np.ones(10), seed=2)
    assert pruned(models, far, pool) == unpruned(models, far, pool) == (0.0, 0)


def _fresh(env_extra, m, seed):
    code = f"""
import json, sys, numpy as np
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, "tests")!r})
import optimobo_b200 as ob
from test_gpu_prune_cascade import problem
models, spec, _, _ = problem()
res = ob.score(models, spec, ob.CandidatePool.counter({m}, np.zeros(10), np.ones(10), seed={seed}), precision="fast")
print(json.dumps([res.best_value, res.best_index]))
"""
    env = dict(os.environ, OMBO_PRUNE_LOG="1", **env_extra)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stderr, tuple(json.loads(out.stdout.strip().splitlines()[-1]))


def test_cascade_against_no_prune_depth1_and_small_caps():
    m, seed = 1 << 22, 11
    err, mine = _fresh({}, m, seed)
    assert "[prune1]" in err and "[prune]" in err                  # both stages ran
    _, off = _fresh({"OMBO_NO_PRUNE": "1"}, m, seed)
    err1, depth1 = _fresh({"OMBO_PRUNE_STAGE1": "0"}, m, seed)
    assert "[prune1]" not in err1 and "[prune]" in err1
    # stage-1 cap: the depth-1 path takes the whole pool; stage-2 cap: the survivors are scored in full
    err_c1, cap1 = _fresh({"OMBO_PRUNE_STAGE1_CAP": "1"}, m, seed)
    assert "[prune1]" in err_c1 and f"[prune] m {m} " in err_c1
    err_c2, cap2 = _fresh({"OMBO_PRUNE_CAP": "1"}, m, seed)
    assert "[prune1]" in err_c2 and "[prune]" in err_c2
    assert mine == off == depth1 == cap1 == cap2
