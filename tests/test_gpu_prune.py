"""GPU: the pruned arg-max of ombo_score (fast mode, exact-semantics 2-D EHVI, only `best` requested).

(a) Preconditions: the BOUND launch of k_posterior_fast8 gives the full launch's mu bit for bit and var_up >= var for
    every candidate (depth 1 and 2, 8 and 16 generator warps, n_pad 256 / 384 / 768 / 1024, ragged m); scoring a
    gathered subset of a pool reproduces the full pool's mu, var and acquisition at those indices bit for bit (the
    survivors are scored that way).
(b) Selection parity: the pruned call returns the same (value, index) as the unpruned fused path -- in process (asking
    for the acquisition values makes a call ineligible) and against OMBO_NO_PRUNE in a fresh process -- over pool
    sizes, seeds, index bases, duplicated candidates, an all-zero pool and a forced-small survivor cap (fallbacks).
(c) Non-eligible calls (reference semantics, requested outputs, FP64, an invalid front, fp16 planes) never enter the
    pruned path (no OMBO_PRUNE_LOG line) and keep their result."""
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


def c5_problem(n=1024, d=10):
    """bench.py's C5 workload (n = 1024; C2 is n = 256): ZDT1, injected hyper-parameters."""
    rng = np.random.default_rng(0)
    X = rng.random((n, d))
    f1 = X[:, 0]
    g = 1 + 9.0 / (d - 1) * X[:, 1:].sum(1)
    Y = np.column_stack([f1, g * (1 - np.sqrt(f1 / g))])
    models = [ob.GPModel(X, Y[:, i], [0.7, 0.8][i] * np.ones(d), [1.0, 2.0][i], device=DEV) for i in range(2)]
    PF, r = ob.host_prep.calc_pf(Y), Y.max(0)
    spec = ob.spec_ehvi(r, PF, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
    return models, spec, PF, r


@pytest.fixture(scope="module")
def c5():
    models, spec, PF, r = c5_problem()
    assert spec.reserved & _cabi.ACQ_FRONT_VALID
    return models, spec, PF, r


def pruned(models, spec, pool):
    res = ob.score(models, spec, pool, precision="fast")
    return res.best_value, res.best_index


def unpruned(models, spec, pool):
    res = ob.score(models, spec, pool, precision="fast", want_acq=True)          # out_acq: not eligible
    return res.best_value, res.best_index, res.acq


def _bound_posterior(model, pool, chunks, gen_warps):
    """mu, var of one model from the BOUND launch (chunks >= 1) or the full one (0), through the library's test hook."""
    lib = _cabi.lib()
    fn = lib.ombo_debug_posterior_bound
    fn.argtypes = [C.c_void_p, C.POINTER(_cabi.Gp), C.POINTER(_cabi.Pool), C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                   C.c_void_p]
    mu = torch.empty(pool.m, dtype=torch.float64, device=DEV)
    var = torch.empty(pool.m, dtype=torch.float64, device=DEV)
    g, p = model.c_struct(1e-15), pool.c_struct()
    ctx = _cabi.Context.get(0)
    _cabi.check(fn(ctx.handle, C.byref(g), C.byref(p), chunks, gen_warps, C.c_void_p(mu.data_ptr()),
                   C.c_void_p(var.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return mu, var


@pytest.mark.parametrize("n", [256, 300, 700, 1024])          # n_pad 256 (C2), 384, 768, 1024 (C5)
def test_bound_mean_is_exact_and_variance_bounds(n):
    models, spec, _, _ = c5_problem(n)
    assert all(m.plane_format == "f8c" for m in models)
    n_chunks = (models[0].n_pad + 255) // 256
    pools = [ob.CandidatePool.counter(m, np.zeros(10), np.ones(10), seed=s) for m, s in ((70001, 3), (1 << 18, 1))]
    pools.append(ob.CandidatePool.explicit(pools[0].rows(0, 4099, DEV).to(torch.float32)))
    for pool in pools:
        full = ob.score(models, spec, pool, precision="fast", want_posterior=True)
        for g, model in enumerate(models):
            for chunks in (1, 2):
                for gw in (8, 16):
                    mu, var = _bound_posterior(model, pool, chunks, gw)
                    assert torch.equal(mu, full.mu[g]), (n, pool.m, g, chunks, gw)
                    assert bool((var >= full.var[g]).all()), (n, pool.m, g, chunks, gw)
                    if chunks >= n_chunks:                          # the bound covers every chunk: it is the variance
                        assert torch.equal(var, full.var[g])
                    elif pool.m > 4099:
                        assert bool((var > full.var[g]).any())


def test_subset_scoring_is_bit_identical(c5):
    models, spec, _, _ = c5
    for m, seed in ((1 << 16, 1), (70001, 5)):
        pool = ob.CandidatePool.counter(m, np.zeros(10), np.ones(10), seed=seed)
        full = ob.score(models, spec, pool, precision="fast", want_posterior=True, want_acq=True)
        rng = np.random.default_rng(seed)
        # random rows, the first / last rows of tiles (128 candidates) and the ragged tail
        idx = np.unique(np.concatenate([rng.choice(m, 300, replace=False), [0, 127, 128, 255, 256, m - 1]]))
        rows = pool.rows(0, m, DEV)[torch.as_tensor(idx, device=DEV)]
        sub = ob.score(models, spec, ob.CandidatePool.explicit(rows), precision="fast", want_posterior=True,
                       want_acq=True)
        it = torch.as_tensor(idx, device=DEV)
        assert torch.equal(sub.mu, full.mu[:, it])
        assert torch.equal(sub.var, full.var[:, it])
        assert torch.equal(sub.acq, full.acq[it])


@pytest.mark.parametrize("m", [1, 63, 257, (1 << 20) + 5, 1 << 24])
def test_selection_parity_sizes(c5, m):
    models, spec, _, _ = c5
    for seed in ((1, 2, 3) if m < (1 << 24) else (1,)):
        pool = ob.CandidatePool.counter(m, np.zeros(10), np.ones(10), seed=seed)
        v, i = pruned(models, spec, pool)
        v_ref, i_ref, _ = unpruned(models, spec, pool)
        assert (v, i) == (v_ref, i_ref), (m, seed)


def test_selection_parity_index_base_and_shards(c5):
    models, spec, _, _ = c5
    pool = ob.CandidatePool.counter(3 << 18, np.zeros(10), np.ones(10), seed=9, index_base=(1 << 33) + 7)
    assert pruned(models, spec, pool) == unpruned(models, spec, pool)[:2]
    for rank in range(3):
        shard = pool.shard(rank, 3)
        assert pruned(models, spec, shard) == unpruned(models, spec, shard)[:2]


def test_duplicates_tie_to_lowest_index(c5):
    models, spec, _, _ = c5
    base = ob.CandidatePool.counter(1 << 16, np.zeros(10), np.ones(10), seed=4)
    _, i_best, _ = unpruned(models, spec, base)
    rows = base.rows(0, 1 << 16, DEV)
    X = torch.cat([rows, rows[i_best:i_best + 1].repeat(5, 1), rows], 0)       # the winner at six indices
    for dtype in (torch.float64, torch.float32):
        pool = ob.CandidatePool.explicit(X.to(dtype))
        v, i = pruned(models, spec, pool)
        assert (v, i) == unpruned(models, spec, pool)[:2]
        if dtype == torch.float64:
            assert i == i_best


def test_all_zero_pool_falls_back(c5):
    models, spec, PF, r = c5
    # a front far ahead of every candidate: every value underflows to 0, the threshold is 0 and nothing is pruned
    far = ob.spec_ehvi(r, PF - 50.0, ob.host_prep.cached_samples(2, 5, seed=0), "exact")
    assert far.reserved & _cabi.ACQ_FRONT_VALID
    pool = ob.CandidatePool.counter(4096, np.zeros(10), np.ones(10), seed=2)
    v, i, acq = unpruned(models, far, pool)
    assert float(acq.max()) == 0.0
    assert pruned(models, far, pool) == (v, i) == (0.0, 0)


def _in_fresh_process(env_extra, m, seed):
    code = f"""
import json, sys, numpy as np
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, "tests")!r})
import optimobo_b200 as ob
from test_gpu_prune import c5_problem
models, spec, _, _ = c5_problem()
res = ob.score(models, spec, ob.CandidatePool.counter({m}, np.zeros(10), np.ones(10), seed={seed}), precision="fast")
print(json.dumps([res.best_value, res.best_index]))
"""
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return out, tuple(json.loads(out.stdout.strip().splitlines()[-1]))


def test_parity_against_no_prune_and_small_cap(c5):
    models, spec, _, _ = c5
    m, seed = 1 << 22, 11
    mine = pruned(models, spec, ob.CandidatePool.counter(m, np.zeros(10), np.ones(10), seed=seed))
    _, off = _in_fresh_process({"OMBO_NO_PRUNE": "1"}, m, seed)
    out, capped = _in_fresh_process({"OMBO_PRUNE_CAP": "1", "OMBO_PRUNE_LOG": "1"}, m, seed)
    assert "[prune]" in out.stderr                                   # the pruned path ran, then fell back
    _, deep = _in_fresh_process({"OMBO_PRUNE_DEPTH": "2"}, m, seed)
    assert mine == off == capped == deep


NON_ELIGIBLE = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import optimobo_b200 as ob
from test_gpu_prune import c5_problem
models, spec, PF, r = c5_problem()
cache = ob.host_prep.cached_samples(2, 5, seed=0)
ref = ob.spec_ehvi(r, PF, cache, "reference")
bad = ob.spec_ehvi(r, np.vstack([PF, PF.max(0)]), cache, "exact")          # a dominated point: not a staircase
pool = ob.CandidatePool.counter(1 << 16, np.zeros(10), np.ones(10), seed=3)
cases = [("eligible", spec, "fast", {{}}), ("reference", ref, "fast", {{}}), ("invalid_front", bad, "fast", {{}}),
         ("fp64", spec, "fp64", {{}}), ("want_acq", spec, "fast", {{"want_acq": True}}),
         ("want_posterior", spec, "fast", {{"want_posterior": True}})]
for name, sp, prec, kw in cases:
    res = ob.score(models, sp, pool, precision=prec, **kw)
    print(name, res.best_value, res.best_index, models[0].plane_format, flush=True)
    sys.stderr.write("== " + name + "\n"); sys.stderr.flush()
"""


def _segments(stderr):
    """OMBO_PRUNE_LOG lines per case: the '== name' marker follows each case's call"""
    seg, cur = {}, []
    for line in stderr.splitlines():
        if line.startswith("== "):
            seg[line[3:]] = cur
            cur = []
        elif line.startswith("[prune]"):
            cur.append(line)
    return seg


def test_non_eligible_calls_stay_off_the_pruned_path(c5):
    code = NON_ELIGIBLE.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    env = dict(os.environ, OMBO_PRUNE_LOG="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    seg = _segments(out.stderr)
    assert len(seg["eligible"]) == 1
    for name in ("reference", "invalid_front", "fp64", "want_acq", "want_posterior"):
        assert seg[name] == [], name
    res = {l.split()[0]: l.split()[1:] for l in out.stdout.splitlines() if l.strip()}
    assert res["eligible"][:2] == res["want_acq"][:2]                # pruned and unpruned agree
    # fp16 planes (OMBO_NO_F8C): never pruned, same result as asking for the values
    out = subprocess.run([sys.executable, "-c", code], env=dict(env, OMBO_NO_F8C="1"), capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert all(v == [] for v in _segments(out.stderr).values())
    res = {l.split()[0]: l.split()[1:] for l in out.stdout.splitlines() if l.strip()}
    assert res["eligible"][2] != "f8c" and res["eligible"][:2] == res["want_acq"][:2]


MAX_UB = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import optimobo_b200 as ob
from test_gpu_prune import c5_problem
models, spec, _, _ = c5_problem()
for seed in range(1, 17):
    res = ob.score(models, spec, ob.CandidatePool.counter(1 << 16, np.zeros(10), np.ones(10), seed=seed), precision="fast")
    print(seed, res.best_value, res.best_index, flush=True)
"""


def test_max_bound_candidate_is_not_always_the_winner(c5):
    """Pools whose largest upper bound belongs to another candidate than the winner: the survivors decide."""
    models, spec, _, _ = c5
    out = subprocess.run([sys.executable, "-c", MAX_UB.format(root=ROOT, tests=os.path.join(ROOT, "tests"))],
                         env=dict(os.environ, OMBO_PRUNE_LOG="1"), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    ub_at = [int(l.split(" at ")[1].split()[0]) for l in out.stderr.splitlines() if l.startswith("[prune]")]
    rows = [l.split() for l in out.stdout.splitlines() if l.strip()]
    assert len(ub_at) == len(rows) == 16
    differ = 0
    for (seed, v, i), at in zip(rows, ub_at):
        pool = ob.CandidatePool.counter(1 << 16, np.zeros(10), np.ones(10), seed=int(seed))
        assert (float(v), int(i)) == unpruned(models, spec, pool)[:2], seed
        differ += int(i) != at
    assert differ >= 1
