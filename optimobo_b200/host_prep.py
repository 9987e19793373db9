"""Candidate-independent, once-per-iteration host preparation for the scoring call
(SURVEY.md section 8a row a13): everything here is O(n^2) or smaller on tiny arrays and feeds
constants to the CUDA kernels.  The reference gets these from pygmo / pymoo
(util_functions.py:64-77,198-199; optimisers.py:182,217-219), neither of which is available.
"""
from __future__ import annotations

import numpy as np
from scipy.stats import norm, qmc


def calc_pf(Y):
    """First non-dominated front (minimisation) in original row order; inputs with fewer than
    two rows are returned unchanged (util_functions.py:64-77)."""
    Y = np.asarray(Y, dtype=np.float64)
    if len(Y) < 2:
        return Y
    le = np.all(Y[:, None, :] <= Y[None, :, :], axis=2)
    lt = np.any(Y[:, None, :] < Y[None, :, :], axis=2)
    dominated = np.any(le & lt, axis=0)
    return Y[~dominated]


def pareto_mask(Y):
    Y = np.asarray(Y, dtype=np.float64)
    le = np.all(Y[:, None, :] <= Y[None, :, :], axis=2)
    lt = np.any(Y[:, None, :] < Y[None, :, :], axis=2)
    return ~np.any(le & lt, axis=0)


def hypervolume(points, ref_point):
    """Exact dominated hypervolume w.r.t. ref_point (minimisation), any k by dimension sweep.
    Stands in for pymoo `HV(ref_point)(Y)` (optimisers.py:217-219) and pygmo
    `hypervolume(PF).compute(r)` (util_functions.py:198-199).  Points beyond the reference
    point contribute nothing."""
    P = np.atleast_2d(np.asarray(points, dtype=np.float64))
    r = np.asarray(ref_point, dtype=np.float64)
    P = P[np.all(P <= r, axis=1)]
    if len(P) == 0:
        return 0.0
    if P.shape[1] == 1:
        return float(r[0] - P[:, 0].min())
    if P.shape[1] == 2:
        Q = P[np.lexsort((P[:, 1], P[:, 0]))]
        total, floor = 0.0, r[1]
        for a, b in Q:
            if b < floor:
                total += (r[0] - a) * (floor - b)
                floor = b
        return float(total)
    Q = P[np.argsort(P[:, -1], kind="stable")]
    total = 0.0
    for i in range(len(Q)):
        top = Q[i + 1, -1] if i + 1 < len(Q) else r[-1]
        if top > Q[i, -1]:
            total += hypervolume(Q[: i + 1, :-1], r[:-1]) * (top - Q[i, -1])
    return float(total)


def ehvi_stripes(PF, ref_point):
    """(2, P+2) array: y1 then y2 of the padded, f2-sorted front (util_functions.py:93-112)."""
    PF = np.atleast_2d(np.asarray(PF, dtype=np.float64))
    S = PF[np.argsort(PF[:, 1])]
    y1 = np.concatenate(([ref_point[0]], S[:, 0], [-np.inf]))
    y2 = np.concatenate(([-np.inf], S[:, 1], [ref_point[1]]))
    return np.stack([y1, y2])


def ehvi_boxes(PF, ref_point):
    """Disjoint boxes tiling {z <= r : no front point dominates z} (minimisation), for the exact EHVI of
    2 <= k <= 4 objectives.  Points not <= r are dropped and the first front is taken; the region is sliced on the
    last objective between consecutive distinct values t_j < z_k <= t_{j+1}, and each slice holds the (k-1)-D
    decomposition for the front of the points with f_k <= t_j.

    Returns (table, boxes):
      table (k, B) float64: row i = [-inf, sorted distinct front coordinates of objective i, r_i], padded with r_i;
      boxes (n_boxes, 2, k) int64 indices into the rows: [c][0] upper, [c][1] lower corner, 0 = -inf.
    An empty front gives the single box [-inf, r]."""
    r = np.asarray(ref_point, dtype=np.float64).reshape(-1)
    k = len(r)
    if not 2 <= k <= 4:
        raise ValueError(f"ehvi_boxes takes 2 to 4 objectives (got {k})")
    P = np.asarray(PF, dtype=np.float64).reshape(-1, k)
    P = calc_pf(P[np.all(P <= r, axis=1)])
    P = np.unique(P, axis=0)
    rows = [np.concatenate(([-np.inf], np.unique(P[:, i]), [r[i]])) for i in range(k)]
    lo, hi = _slice_boxes(P, r)
    boxes = np.empty((len(lo), 2, k), dtype=np.int64)
    for i in range(k):
        boxes[:, 0, i] = np.searchsorted(rows[i], hi[:, i], side="left")
        boxes[:, 1, i] = np.searchsorted(rows[i], lo[:, i], side="left")
    B = max(len(row) for row in rows)
    table = np.stack([np.concatenate((row, np.full(B - len(row), r[i]))) for i, row in enumerate(rows)])
    return table, boxes


def _slice_boxes(P, r):
    """(lower, upper) corners, each (n_boxes, k), of the decomposition ehvi_boxes describes; P is a front <= r."""
    k = len(r)
    if k == 2:
        # slice j of f2 between t_j and t_{j+1}: f1 is free up to the least f1 of the points with f2 <= t_j
        t = np.unique(P[:, 1])
        edges = np.concatenate(([-np.inf], t, [r[1]]))
        S = P[np.argsort(P[:, 1], kind="stable")]
        run = np.minimum.accumulate(S[:, 0]) if len(S) else S[:, 0]
        last = np.searchsorted(S[:, 1], t, side="right") - 1          # last point with f2 <= t_j
        right = np.concatenate(([r[0]], run[last]))
        keep = edges[1:] > edges[:-1]
        lo = np.column_stack([np.full(keep.sum(), -np.inf), edges[:-1][keep]])
        hi = np.column_stack([right[keep], edges[1:][keep]])
        return lo, hi
    t = np.unique(P[:, -1])
    edges = np.concatenate(([-np.inf], t, [r[-1]]))
    los, his = [], []
    for j in range(len(edges) - 1):
        if edges[j + 1] <= edges[j]:
            continue
        sub = calc_pf(P[P[:, -1] <= edges[j], :-1])
        lo, hi = _slice_boxes(sub, r[:-1])
        los.append(np.column_stack([lo, np.full(len(lo), edges[j])]))
        his.append(np.column_stack([hi, np.full(len(hi), edges[j + 1])]))
    return np.concatenate(los), np.concatenate(his)


def cache_covariance(cache):
    """(C00, C01) of np.cov(cache[:,0], cache[:,1]); the reference's EHVI passes
    var0*C00, var0*C01 as 'sigma' (util_functions.py:163,167; SURVEY section 0.4)."""
    c = np.cov(np.asarray(cache)[:, 0], np.asarray(cache)[:, 1])
    return float(c[0, 0]), float(c[0, 1])


def decompose_into_cells(pf, ideal_point, max_point):
    """Cells of the non-dominated region of a 2-D front as (n_cells, 2, 2) with [c][0] = upper
    and [c][1] = lower corner -- the staircase the reference's WFG-style walk produces
    (emo.py:55-152, util_functions.py:414-517), built directly from the f1-sorted front."""
    pf = np.atleast_2d(np.asarray(pf, dtype=np.float64))
    if pf.shape[1] != 2:
        raise ValueError("cell decomposition is 2-D only (emo.py:21)")
    S = pf[np.argsort(pf[:, 0], kind="stable")]
    n = len(S)
    cells = np.empty((n + 1, 2, 2))
    cells[0, 0] = (S[0, 0], max(S[0, 1], max_point[1]))
    cells[0, 1] = ideal_point
    for c in range(1, n + 1):
        right = S[c, 0] if c < n else max(S[-1, 0], max_point[0])
        cells[c, 0] = (right, S[c - 1, 1])
        cells[c, 1] = (S[c - 1, 0], ideal_point[1])
    return cells


def get_reference_directions(name, n_dim, n_partitions):
    """pymoo's das-dennis simplex lattice (optimisers.py:182,453; parego.py:167; ...)."""
    if name != "das-dennis":
        raise ValueError("only 'das-dennis' reference directions are provided")
    rows = []
    stack = [((), n_partitions)]
    while stack:
        prefix, left = stack.pop()
        if len(prefix) == n_dim - 1:
            rows.append(prefix + (left,))
            continue
        for i in range(left, -1, -1):
            stack.append((prefix + (i,), left - i))
    return np.asarray(rows, dtype=np.float64) / n_partitions


def latin_hypercube(num_samples, variable_ranges, rng=None):
    """One stratified, independently permuted sample per variable (util_functions.py:46-61).
    Like the reference, the in-stratum offset is (k + u)/n of the stratum width (its `points`
    are already divided by n before being scaled by the stratum width), i.e. samples sit in the
    lower part of each stratum."""
    rng = np.random.default_rng() if rng is None else rng
    n = num_samples
    out = np.empty((n, len(variable_ranges)))
    for j, (lo, hi) in enumerate(variable_ranges):
        width = (hi - lo) / n
        frac = (rng.random(n) + np.arange(n)) / n
        out[:, j] = rng.permutation(lo + width * np.arange(n) + width * frac)
    return out


def cached_samples(n_obj, sample_exponent, seed=None):
    """2**sample_exponent scrambled-Sobol points pushed through the normal quantile
    (optimisers.py:121-141)."""
    pts = qmc.Sobol(d=n_obj, scramble=True, seed=seed).random_base2(m=sample_exponent)
    return norm.ppf(pts)
