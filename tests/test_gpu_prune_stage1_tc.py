"""GPU: stage 1 of the pruned arg-max on the tensor core (posterior_stage1_tc.cu).

(a) The certified margin: |mu~ - mu_F| <= M for every candidate, mu_F the full f8c launch's FP32 mean (n_pad 256 / 384 /
    768 / 1024, d 1..12, Matern and RBF pairs, counter / f32 / f64 pools, ragged m, candidates equal to training rows);
    the largest ratio is printed and must stay below 1/4 (the margin carries a safety factor of 4).
(b) Its bound is >= the full value of every candidate up to the FP32 contract; the largest bound and its index.
(c) The cascade on its default stage 1 returns what the mean8 stage 1 (OMBO_STAGE1_KERNEL=mean8), the depth-1 path
    alone and the unpruned call return; at a short length-scale the default stage 1 is the exact-mean kernel."""
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
from test_gpu_prune_cascade import ROOT, _fresh, pools, problem  # noqa: E402

DEV = "cuda:0"
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cabi.fast_path_available(), reason="fast path not built")]
RATIOS = []


def stage1_tc(models, spec, pool):
    """mu~ [2, m], M [2, m], UB [m] and the largest bound of the tensor-core stage-1 launch (test hook)."""
    fn = _cabi.lib().ombo_debug_stage1_tc
    fn.argtypes = [C.c_void_p, C.POINTER(_cabi.Gp), C.POINTER(_cabi.Pool), C.POINTER(_cabi.Acq)] + [C.c_void_p] * 5
    mu = torch.empty((2, pool.m), dtype=torch.float64, device=DEV)
    marg = torch.empty((2, pool.m), dtype=torch.float64, device=DEV)
    ub = torch.empty(pool.m, dtype=torch.float64, device=DEV)
    best = torch.empty(2, dtype=torch.int64, device=DEV)
    gps = (_cabi.Gp * 2)(*[m.c_struct(1e-15) for m in models])
    p, a = pool.c_struct(), spec.c_struct(torch.device(DEV))
    ctx = _cabi.Context.get(0)
    _cabi.check(fn(ctx.handle, gps, C.byref(p), C.byref(a), *[C.c_void_p(t.data_ptr()) for t in (mu, marg, ub, best)],
                   C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return mu, marg, ub, best


def check_margin(models, spec, pool, tag):
    full = ob.score(models, spec, pool, precision="fast", want_posterior=True, want_acq=True)
    mu, marg, ub, _ = stage1_tc(models, spec, pool)
    assert bool(torch.isfinite(mu).all()) and bool((marg > 0).all()), tag
    ratio = float(((mu - full.mu).abs() / marg).max())
    RATIOS.append((tag, ratio))
    print(f"max |mu~ - mu_F| / M {ratio:.3g} at {tag}")
    assert ratio <= 1.0 / 4, tag                                   # the derivation carries a safety factor of 4
    # the bound: never below the full value beyond the FP32 contract of the acquisition (NaN: the candidate survives)
    ok = torch.isnan(ub) | (ub >= full.acq - 2e-3 * float(ub[~torch.isnan(ub)].max()))
    assert bool(ok.all()), tag


@pytest.mark.parametrize("n", [256, 300, 700, 1024])          # n_pad 256, 384, 768, 1024
def test_stage1_tc_margin_n_pad(n):
    models, spec, _, _ = problem(n)
    for pool in pools(10, 70001):
        check_margin(models, spec, pool, ("n", n, pool.m))


@pytest.mark.parametrize("d", list(range(1, 13)))
@pytest.mark.parametrize("kernels", [("matern52", "matern52"), ("rbf", "rbf"), ("matern52", "rbf"), ("rbf", "matern52")])
def test_stage1_tc_margin_d_kernel(d, kernels):
    models, spec, _, _ = problem(300, d, kernels, noise=2e-2)
    for pool in pools(d, 4099):
        check_margin(models, spec, pool, ("d", d, kernels))


def test_stage1_tc_margin_training_rows():
    # candidates on the training points (r^2 -> 0, where the FP32 chains may round r^2 below zero), and next to them
    models, spec, _, _ = problem(700)
    Xt = torch.as_tensor(np.random.default_rng(0).random((700, 10)), device=DEV)      # problem()'s training inputs
    rows = torch.cat([Xt, Xt + 1e-7, Xt[:5].repeat(3, 1)], 0)
    for dtype in (torch.float64, torch.float32):
        check_margin(models, spec, ob.CandidatePool.explicit(rows.to(dtype)), ("train", str(dtype)))


def test_stage1_tc_largest_bound():
    models, spec, _, _ = problem()
    pool = ob.CandidatePool.counter(100003, np.zeros(10), np.ones(10), seed=5, index_base=1 << 33)
    _, _, ub, best = stage1_tc(models, spec, pool)
    w = torch.where(torch.isnan(ub), torch.full_like(ub, -np.inf), ub)
    assert best[:1].view(torch.float64).item() == float(w.max())
    assert int(best[1]) == (1 << 33) + int(torch.nonzero(w == w.max())[0])


@pytest.mark.parametrize("m,seed", [(1 << 22, 11), (1 << 24, 1)])
def test_stage1_tc_cascade_against_mean8_depth1_and_unpruned(m, seed):
    err, tc = _fresh({}, m, seed)
    assert "[prune1]" in err and "[prune]" in err and "stage1 tc" in err        # the tensor-core kernel ran
    err8, mean8 = _fresh({"OMBO_STAGE1_KERNEL": "mean8"}, m, seed)
    assert "[prune1]" in err8 and "stage1 mean8" in err8
    _, depth1 = _fresh({"OMBO_PRUNE_STAGE1": "0"}, m, seed)
    _, off = _fresh({"OMBO_NO_PRUNE": "1"}, m, seed)
    assert tc == mean8 == depth1 == off
    s_tc = int(err.split("[prune1] m")[1].split("survivors")[1].split()[0])
    s_8 = int(err8.split("[prune1] m")[1].split("survivors")[1].split()[0])
    print(f"stage-1 survivors at m {m}: tensor core {s_tc}, mean8 {s_8}")
    assert s_tc <= 2 * s_8                       # measured 1.66x (2^22, seed 11) and 1.32x (2^24, seed 1)


SHORT = '''
import json, sys, numpy as np
sys.path.insert(0, {root!r})
import optimobo_b200 as ob
rng = np.random.default_rng(0)
X = rng.random((1024, 10))
f1 = X[:, 0]
g = 1 + X[:, 1:].sum(1)
Y = np.column_stack([f1, g * (1 - np.sqrt(f1 / g))])
models = [ob.GPModel(X, Y[:, i], {ell} * np.ones(10), [1.0, 2.0][i], kernel="matern52", device="cuda:0") for i in range(2)]
assert all(m.plane_format == "f8c" for m in models)
spec = ob.spec_ehvi(Y.max(0), ob.host_prep.calc_pf(Y), ob.host_prep.cached_samples(2, 5, seed=0), "exact")
pool = ob.CandidatePool.counter(1 << 20, np.zeros(10), np.ones(10), seed=3)
res = ob.score(models, spec, pool, precision="fast")
ref = ob.score(models, spec, pool, precision="fast", want_acq=True)
print(json.dumps([res.best_value, res.best_index, ref.best_value, ref.best_index]))
'''


def _short(ell, env_extra):
    env = dict(os.environ, OMBO_PRUNE_LOG="1", **env_extra)
    out = subprocess.run([sys.executable, "-c", SHORT.format(root=ROOT, ell=ell)], env=env, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    v = json.loads(out.stdout.strip().splitlines()[-1])
    assert v[:2] == v[2:]                        # the pruned call returns the unpruned call's (value, index)
    line = [ln for ln in out.stderr.splitlines() if ln.startswith("[prune1]")][0]
    return line, int(line.split("survivors")[1].split()[0])


def test_stage1_short_length_scale_keeps_the_exact_mean_stage():
    # at ell = 0.03 the pool's T is far past where the margin prunes well: the default stage 1 is the exact-mean kernel,
    # with the mean8 arm's survivors; at the C5 length-scale it is the tensor-core kernel
    line, n = _short(0.03, {})
    line8, n8 = _short(0.03, {"OMBO_STAGE1_KERNEL": "mean8"})
    print(line, line8, sep="\n")
    assert "stage1 mean8" in line and n == n8
    line, _ = _short(0.7, {})
    assert "stage1 tc" in line
