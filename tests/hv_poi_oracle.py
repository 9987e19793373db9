"""CPU oracles of the hypervolume-based probability of improvement for 2 to 4 objectives (numpy / scipy, float64),
the value OMBO_ACQ_HV_POI_BOX computes.  Only the tests import it.

For a front PF, an ideal point and a max point, R = {ideal <= z <= r' : no front point p <= z} with
r' = max(max_point, PF.max(0)) per objective, and for y_i ~ N(mu_i, var_i + 1e-5) independent:
    value = P(y in R) * vol(R above mu).
Both oracles sum disjoint cells of R: `hv_poi_box_batched` the boxes of host_prep.ehvi_boxes with the table clamped
below at the ideal point, `hv_poi_grid_batched` every cell of the full breakpoint grid that no front point dominates
(it never builds boxes; its cost is (B - 1)^k cells per candidate).  A cell's probability mass is taken as the
difference of two lower tails below the mean and of two upper tails above it, so that neither oracle cancels far
from the mean."""
from __future__ import annotations

import numpy as np
from scipy.special import ndtr

VAR_EPS = 1e-5


def _mass(lo, hi, mu, sd):
    """P(lo < y <= hi) for y ~ N(mu, sd^2), elementwise, without subtracting two numbers near 1."""
    with np.errstate(all="ignore"):
        zl, zu = (lo - mu) / sd, (hi - mu) / sd
        return np.where(zl > 0, ndtr(-zl) - ndtr(-zu), ndtr(zu) - ndtr(zl))


def _extent(lo, hi, mu):
    """Length of [lo, hi] above mu: max(hi - max(lo, mu), 0)."""
    return np.clip(hi - np.maximum(lo, mu), 0.0, None)


def region_ref(PF, max_point):
    """r' = max(max_point, PF.max(0)) per objective (max_point for an empty front)."""
    r = np.asarray(max_point, float).reshape(-1)
    P = np.asarray(PF, float).reshape(-1, len(r))
    return np.maximum(r, P.max(0)) if len(P) else r


def hv_poi_box_batched(mu, var, PF, ideal, max_point):
    """PoI * Imp over the boxes of host_prep.ehvi_boxes(PF, r'), breakpoints clamped below at the ideal point.
    mu, var: (m, k).  Returns (m,)."""
    from optimobo_b200 import host_prep
    mu = np.atleast_2d(np.asarray(mu, float))
    sd = np.sqrt(np.atleast_2d(np.asarray(var, float)) + VAR_EPS)
    ideal = np.asarray(ideal, float).reshape(-1)
    table, boxes = host_prep.ehvi_boxes(PF, region_ref(PF, max_point))
    table = np.maximum(table, ideal[:, None])
    poi = np.ones((len(mu), len(boxes)))
    imp = np.ones((len(mu), len(boxes)))
    for i in range(len(ideal)):
        U, L = table[i, boxes[:, 0, i]][None, :], table[i, boxes[:, 1, i]][None, :]
        poi *= _mass(L, U, mu[:, i:i + 1], sd[:, i:i + 1])
        imp *= _extent(L, U, mu[:, i:i + 1])
    return poi.sum(1) * imp.sum(1)


def hv_poi_grid_batched(mu, var, PF, ideal, max_point):
    """The same value by brute force: grid row i = the distinct values of ideal_i, r'_i and the front's coordinates
    between them; a cell is in R iff no front point p <= its lower corner.  mu, var: (m, k).  Returns (m,)."""
    mu = np.atleast_2d(np.asarray(mu, float))
    sd = np.sqrt(np.atleast_2d(np.asarray(var, float)) + VAR_EPS)
    ideal = np.asarray(ideal, float).reshape(-1)
    r = region_ref(PF, max_point)
    k = len(r)
    P = np.asarray(PF, float).reshape(-1, k)
    hi = np.maximum(r, ideal)
    grid = [np.unique(np.clip(np.concatenate(([ideal[i], hi[i]], P[:, i])), ideal[i], hi[i])) for i in range(k)]
    shape = tuple(len(g) - 1 for g in grid)
    dominated = np.zeros(shape, dtype=bool)
    for p in P:
        sl = tuple(slice(int(np.searchsorted(grid[i][:-1], p[i], side="left")), None) for i in range(k))
        dominated[sl] = True
    free = (~dominated).astype(float)

    def contract(per_obj):
        acc = np.einsum("...c,mc->m...", free, per_obj[-1])
        for i in range(k - 2, -1, -1):
            acc = np.einsum("m...c,mc->m...", acc, per_obj[i])
        return acc

    lo = [g[None, :-1] for g in grid]
    up = [g[None, 1:] for g in grid]
    poi = contract([_mass(lo[i], up[i], mu[:, i:i + 1], sd[:, i:i + 1]) for i in range(k)])
    imp = contract([_extent(lo[i], up[i], mu[:, i:i + 1]) for i in range(k)])
    return poi * imp
