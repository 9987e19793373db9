"""Host side of the pruned arg-max of ombo_score (fast mode, exact-semantics 2-D EHVI).  No GPU needed.

* The property the pruning rests on: over a valid staircase front the exact 2-D EHVI (oracle, FP64) never decreases
  as either objective's sigma grows, from sigma -> 0 to deep in the tails.
* A CPU simulation of the rule (upper bound from the first 256 training points, keep UB >= v0 - tau) picks the same
  (value, index) as the full arg-max.
* The BOUND schedule of the f8c kernel (posterior_fast8.cu::f8_build_schedule): every block generated once, in order;
  the bounded chunks take exactly the full schedule's steps; no store or reload; MEAN on exactly the other blocks.
* host_prep.front_is_staircase and the bit spec_ehvi sets from it."""
import ctypes
import os
import sys

import numpy as np
import pytest
import scipy.linalg as sla

from optimobo_b200 import _cabi, host_prep
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TAU = 2e-3             # OMBO_PRUNE_TAU (api.cu)


def staircase(rng, p):
    f1 = np.sort(rng.random(p))[::-1]
    f2 = np.sort(rng.random(p))
    return np.column_stack([f1, f2]), np.array([1.2, 1.3])


@pytest.mark.parametrize("seed", range(6))
def test_exact_ehvi_non_decreasing_in_sigma(seed):
    rng = np.random.default_rng(seed)
    PF, r = staircase(rng, int(rng.integers(1, 40)))
    assert host_prep.front_is_staircase(PF, r)
    m = 400
    # means around the front, behind it (deep tails) and beyond the reference point
    mu = np.concatenate([rng.uniform(-0.5, 1.8, (m, 2)), rng.uniform(3.0, 9.0, (m // 4, 2))])
    sig = np.geomspace(1e-6, 30.0, 60)
    for obj in (0, 1):
        other = rng.uniform(0.01, 1.0, len(mu))
        prev = None
        for s in sig:
            s0 = np.full(len(mu), s) if obj == 0 else other
            s1 = other if obj == 0 else np.full(len(mu), s)
            v = O.ehvi_batched(mu[:, 0], mu[:, 1], s0 ** 2, s1 ** 2, PF, r, None, "exact")
            assert np.all(np.isfinite(v)) and np.all(v >= 0)
            if prev is not None:
                # FP64 rounding only: relative 1e-12 of the value
                assert np.all(v >= prev - 1e-12 * np.abs(prev) - 1e-300), (obj, s)
            prev = v


def test_pruning_simulation_matches_full_argmax():
    sys.path.insert(0, ROOT)
    import bench as B
    X, Y, ells, sf2 = B.workload()
    st = [O.gp_fit_state(X, Y[:, i], ells[i], sf2[i]) for i in range(2)]
    PF, r = O.calc_pf(Y), Y.max(0)
    for seed, m in ((1, 4096), (2, 3000)):
        Xc = O.candidates_from_counter(seed, 0, m, np.zeros(10), np.ones(10))
        mus, var, vup = [], [], []
        for S in st:
            Kx = O.k_of_r(O.scaled_dist(S["X"], Xc, S["ell"], S["form"]), S["sigma_f2"], S["kernel"])
            mus.append(Kx.T @ S["alpha"])
            V = sla.solve_triangular(S["L"], Kx, lower=True, check_finite=False)
            c = np.cumsum(np.square(V), 0)
            var.append(np.clip(S["sigma_f2"] - c[-1], 1e-15, None))
            vup.append(np.clip(S["sigma_f2"] - c[255], 1e-15, None))
        assert np.all(vup[0] >= var[0]) and np.all(vup[1] >= var[1])
        val = O.ehvi_batched(mus[0], mus[1], var[0], var[1], PF, r, None, "exact")
        ub = O.ehvi_batched(mus[0], mus[1], vup[0], vup[1], PF, r, None, "exact")
        i_max = int(np.argmax(ub))
        v0 = val[i_max]
        keep = np.flatnonzero(np.isnan(ub) | (ub >= v0 - TAU * ub[i_max]))
        assert len(keep) < m // 20
        j = int(np.argmax(val[keep]))
        best = max((val[keep][j], -int(keep[j])), (v0, -i_max))
        assert (best[0], -best[1]) == (val.max(), int(np.argmax(val)))


def _bound_schedule(n_pad, chunks):
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    buf = np.zeros(1 << 12, np.uint32)
    for name, args in (("ombo_debug_f8_bound_schedule", (n_pad, chunks)), ("ombo_debug_f8_schedule", (n_pad, 3.0, 0))):
        fn = getattr(lib, name)
        fn.argtypes = [ctypes.c_int] + ([ctypes.c_int] if len(args) == 2 else [ctypes.c_double, ctypes.c_int]) + \
                      [ctypes.c_void_p, ctypes.c_int]
        n = fn(*args, buf.ctypes.data, buf.size)
        assert 0 < n <= buf.size
        if name == "ombo_debug_f8_bound_schedule":
            bound = [int(w) for w in buf[:n]]
        else:
            full = [int(w) for w in buf[:n]]
    return bound, full


@pytest.mark.parametrize("chunks", [1, 2])
@pytest.mark.parametrize("n_pad", [128, 256, 384, 512, 640, 1024, 1152, 2048, 8192])
def test_bound_schedule_invariants(n_pad, chunks):
    bound, full = _bound_schedule(n_pad, chunks)
    nkb = n_pad // 64
    nb = min(nkb, 4 * chunks)
    assert [w & 0xFF for w in bound] == list(range(nkb)), "every block generated once, in order"
    for w in bound:
        assert (w >> 8) & 1 and not (w >> 9) & 1, "fresh, never stored"
        mean = (w >> 26) & 1
        assert mean == ((w & 0xFF) >= nb), "MEAN exactly beyond the bound"
        if mean:
            assert ((w >> 10) & 0xFFF) == 0 and ((w >> 22) & 0xF) == 0, "a MEAN step multiplies nothing"
    # the bounded chunks: the same steps (block, slot, N, FIRST / DONE) in the same order as the full schedule
    def chunk_steps(steps, c):
        out = []
        for w in steps:
            for s in (0, 1):
                if ((w >> (10 + 6 * s)) & 63) - 1 == c:
                    out.append((w & 0xFF, (w >> 8) & 1, s, (w >> (22 + s)) & 1, (w >> (24 + s)) & 1))
        return out
    for c in range(min(chunks, (n_pad + 255) // 256)):
        assert chunk_steps(bound, c) == chunk_steps(full, c)
    assert all(((w >> (10 + 6 * s)) & 63) - 1 < chunks for w in bound for s in (0, 1))


def test_front_is_staircase():
    r = np.array([1.0, 1.0])
    good = np.array([[0.1, 0.9], [0.5, 0.5], [0.9, 0.1]])
    assert host_prep.front_is_staircase(good, r)
    assert host_prep.front_is_staircase(good[::-1], r)                       # any input order
    assert host_prep.front_is_staircase(np.array([[1.0, 1.0]]), r)            # on the reference point
    assert not host_prep.front_is_staircase(np.vstack([good, [0.6, 0.6]]), r)  # dominated
    assert not host_prep.front_is_staircase(np.vstack([good, good[:1]]), r)    # duplicate
    assert not host_prep.front_is_staircase(np.vstack([good, [1.1, 0.0]]), r)  # beyond r
    assert not host_prep.front_is_staircase(np.array([[np.nan, 0.5]]), r)
    from optimobo_b200.acquisition import spec_ehvi
    cache = host_prep.cached_samples(2, 5, seed=0)
    assert spec_ehvi(r, good, cache, "exact").reserved == _cabi.ACQ_FRONT_VALID
    assert spec_ehvi(r, np.vstack([good, [0.6, 0.6]]), cache, "exact").reserved == 0
