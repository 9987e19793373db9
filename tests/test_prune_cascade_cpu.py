"""Host side of the two-stage pruned arg-max (stage 1: the mean-only bound of posterior_mean8.cu).  No GPU needed.

A CPU simulation on the oracle (C5 workload of bench.py): stage 1 bounds every candidate with its exact mean and the
prior variance, takes the threshold from the full scores of the largest bounds of T blocks of the pool (the per-CTA
maxima of the launch) and keeps UB1 >= v0 - tau UB1_max; stage 2 runs the depth-1 rule (chunk-0 bound, the first 256
training points) on the survivors.  The result is the full arg-max for any T, and with more than one block stage 1
keeps a small share of the pool."""
import os
import sys

import numpy as np
import scipy.linalg as sla

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TAU = 2e-3             # OMBO_PRUNE_TAU (api.cu)


def _depth1(val, ub):
    """the depth-1 rule on a candidate set: (best value, local index), survivors"""
    i_max = int(np.argmax(np.where(np.isnan(ub), -np.inf, ub)))
    v0 = val[i_max]
    keep = np.flatnonzero(np.isnan(ub) | (ub >= v0 - TAU * ub[i_max]))
    j = int(np.argmax(val[keep]))
    best = max((val[keep][j], -int(keep[j])), (v0, -i_max))
    return (best[0], -best[1]), len(keep)


def test_cascade_simulation_matches_full_argmax():
    sys.path.insert(0, ROOT)
    import bench as B
    X, Y, ells, sf2 = B.workload()
    st = [O.gp_fit_state(X, Y[:, i], ells[i], sf2[i]) for i in range(2)]
    PF, r = O.calc_pf(Y), Y.max(0)
    for seed, m, n_top in ((1, 8192, 16), (2, 6000, 1), (3, 8192, 148)):
        Xc = O.candidates_from_counter(seed, 0, m, np.zeros(10), np.ones(10))
        mus, var, vup, vprior = [], [], [], []
        for S in st:
            Kx = O.k_of_r(O.scaled_dist(S["X"], Xc, S["ell"], S["form"]), S["sigma_f2"], S["kernel"])
            mus.append(Kx.T @ S["alpha"])
            V = sla.solve_triangular(S["L"], Kx, lower=True, check_finite=False)
            c = np.cumsum(np.square(V), 0)
            var.append(np.clip(S["sigma_f2"] - c[-1], 1e-15, None))
            vup.append(np.clip(S["sigma_f2"] - c[255], 1e-15, None))
            vprior.append(np.full(m, S["sigma_f2"]))
        val = O.ehvi_batched(mus[0], mus[1], var[0], var[1], PF, r, None, "exact")
        ub1 = O.ehvi_batched(mus[0], mus[1], vprior[0], vprior[1], PF, r, None, "exact")
        ub2 = O.ehvi_batched(mus[0], mus[1], vup[0], vup[1], PF, r, None, "exact")
        assert np.all(ub1 >= ub2 - 1e-12 * np.abs(ub2)) and np.all(ub2 >= val - 1e-12 * np.abs(val))
        # stage 1: threshold from the best full score among the largest bounds of n_top blocks
        top = np.array([b[int(np.argmax(ub1[b]))] for b in np.array_split(np.arange(m), n_top)])
        t = int(np.argmax(val[top]))
        v0, i0 = val[top[t]], int(top[t])
        keep1 = np.flatnonzero(np.isnan(ub1) | (ub1 >= v0 - TAU * ub1.max()))
        if n_top > 1:                      # the bound arg-max alone can score far below the pool's best
            assert len(keep1) < m // 8
        # stage 2: the depth-1 rule on the survivors, indices mapped back
        (v2, j2), n2 = _depth1(val[keep1], ub2[keep1])
        best = max((v2, -int(keep1[j2])), (v0, -i0))
        assert (best[0], -best[1]) == (val.max(), int(np.argmax(val)))
        assert n2 <= len(keep1)
