#!/usr/bin/env python
"""How many candidates a variance bound leaves for the exact arg-max of the C5 pool (CPU, FP64 oracle; math, no timing).

For each candidate: the exact mean, the posterior variance and the upper bound sigma_f2 - sum_{j<t} V_ij^2 from the
first t training points (L^-1 is lower triangular, so that sum is the variance reduction of those points alone).  The
exact 2-D EHVI never decreases in either sigma over a valid front, so the EHVI at the bounds is an upper bound UB;
the script counts the candidates whose UB reaches the pool's best value (with margins 1, 1.01, 1.1).
t = 256 is chunk 0 of the f8c kernel (OMBO_PRUNE_DEPTH=1), t = 512 pass 0 (OMBO_PRUNE_DEPTH=2).

usage: python scripts/prune_study.py [log2 m (default 16)] [pool seed (default 1)]"""
import os
import sys

import numpy as np
import scipy.linalg as sla

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
import bench as B  # noqa: E402

TS = (0, 64, 128, 256, 512)


def main():
    log2m = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    X, Y, ells, sf2 = B.workload()
    st = [O.gp_fit_state(X, Y[:, i], ells[i], sf2[i]) for i in range(2)]
    PF, r = O.calc_pf(Y), Y.max(0)
    M, chunk = 1 << log2m, 8192
    mus = [np.empty(M) for _ in range(2)]
    vs = {t: [np.empty(M) for _ in range(2)] for t in TS + (None,)}
    for s in range(0, M, chunk):
        c = min(chunk, M - s)
        Xc = O.candidates_from_counter(seed, s, c, np.zeros(10), np.ones(10))
        for g, S in enumerate(st):
            Kx = O.k_of_r(O.scaled_dist(S["X"], Xc, S["ell"], S["form"]), S["sigma_f2"], S["kernel"])
            mus[g][s:s + c] = Kx.T @ S["alpha"]
            V = sla.solve_triangular(S["L"], Kx, lower=True, check_finite=False)
            cs = np.concatenate([np.zeros((1, c)), np.cumsum(np.square(V), 0)])
            for t in vs:
                vs[t][g][s:s + c] = np.clip(S["sigma_f2"] - cs[-1 if t is None else t], 1e-15, None)
    e = {t: O.ehvi_batched(mus[0], mus[1], vs[t][0], vs[t][1], PF, r, None, "exact") for t in vs}
    best = e[None].max()
    print(f"pool 2^{log2m} seed {seed}: best {best:.6g} at {int(e[None].argmax())}")
    for t in TS:
        assert np.all(e[t] >= e[None] * (1 - 1e-9)), "bound below the value"
        n = [int((e[t] * k >= best).sum()) for k in (1.0, 1.01, 1.1)]
        ratio = np.sqrt(vs[t][0] / vs[None][0])
        print(f"t = {t:4d}: survivors (margin 1 / 1.01 / 1.1) {n}, fraction {n[1] / M:.2e}; "
              f"sigma_up / sigma of model 0: median {np.median(ratio):.3f}")


if __name__ == "__main__":
    main()
