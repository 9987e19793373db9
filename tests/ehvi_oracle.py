"""CPU oracle of the exact k-objective EHVI (numpy / scipy, float64), independent of optimobo_b200.host_prep: it
never builds boxes.  It sums over every cell of the full breakpoint grid and skips the cells a front point
dominates, so its cost is (B - 1)^k cells per candidate.  Only the tests import it."""
from __future__ import annotations

import numpy as np
from scipy.special import ndtr

_NORM_PDF_C = np.sqrt(2.0 * np.pi)


def expected_shortfall(t, mu, sd):
    """H(t) = E[(t - y)^+] for y ~ N(mu, sd^2), elementwise; H(-inf) = 0."""
    t, mu, sd = np.broadcast_arrays(np.asarray(t, float), np.asarray(mu, float), np.asarray(sd, float))
    out = np.zeros(t.shape)
    fin = np.isfinite(t)
    with np.errstate(all="ignore"):
        z = (t[fin] - mu[fin]) / sd[fin]
        out[fin] = (t[fin] - mu[fin]) * ndtr(z) + sd[fin] * np.exp(-0.5 * z * z) / _NORM_PDF_C
    return out


def ehvi_grid_batched(mu, var, PF, r):
    """Exact EHVI of m candidates with independent objectives y_i ~ N(mu[:, i], var[:, i]) against the front PF
    (minimisation) and reference point r.  Grid row i = [-inf, sorted distinct coordinates of objective i of the
    points <= r, r_i]; a cell is dominated iff some point p <= its lower corner; EHVI = sum over the other cells of
    prod_i (H_i(upper_i) - H_i(lower_i)).  mu, var: (m, k).  Returns (m,)."""
    mu = np.atleast_2d(np.asarray(mu, float))
    sd = np.sqrt(np.atleast_2d(np.asarray(var, float)))
    r = np.asarray(r, float).reshape(-1)
    k = len(r)
    P = np.asarray(PF, float).reshape(-1, k)
    P = P[np.all(P <= r, axis=1)]
    grid = [np.concatenate(([-np.inf], np.unique(np.concatenate((P[:, i], [r[i]]))))) for i in range(k)]
    shape = tuple(len(g) - 1 for g in grid)
    # dominated cells: lower corner >= p in every objective, for some p
    dominated = np.zeros(shape, dtype=bool)
    for p in P:
        sl = tuple(slice(int(np.searchsorted(grid[i][:-1], p[i], side="left")), None) for i in range(k))
        dominated[sl] = True
    free = (~dominated).astype(float)
    # per objective: D_i[m, j] = H_i(grid_i[j + 1]) - H_i(grid_i[j])
    D = []
    for i in range(k):
        Hg = expected_shortfall(grid[i][None, :], mu[:, i:i + 1], sd[:, i:i + 1])
        D.append(Hg[:, 1:] - Hg[:, :-1])
    # contract the cell mask with the D_i one objective at a time: acc[m, j_1 .. j_l]
    acc = np.einsum("...c,mc->m...", free, D[-1])
    for i in range(k - 2, -1, -1):
        acc = np.einsum("m...c,mc->m...", acc, D[i])
    return acc
