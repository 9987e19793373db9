"""Host side of the tensor-core stage 1 of the pruned arg-max (posterior_stage1_tc.cu).  No GPU needed.

* The FMA-pipe 2^t of the consumers (s1_exp2_poly): every FP32 reduced argument f with 2^-12 <= |f| <= 0.5 and a dense
  sample below, within 2^-21 of 2^f; the exponent insertion over t in [-125, 0] and the clamp below.
* A float32 / float16 restatement of both distance paths (the full launch's FP32 chain, the fp16 hi / lo split with the
  norm columns) against the r^2 bounds of the margin, on random and adversarial inputs (training rows as candidates,
  extreme length-scales, large |x|), and the margin M against |mu~ - mu_F| computed from them.
* The monotonicity the margin rests on: the exact 2-D EHVI (oracle, FP64) never decreases as either mean decreases."""
import numpy as np
import pytest

from oracle import oracle as O

U = 2.0 ** -24
G_F, G_TC, E_SUB, ETA, ETA_ABS, SAFETY = 13.0, 56.0, 7.0 * U, 48.0 * U, 32.0 * U, 4.0   # posterior_stage1_tc.cu
C = np.array([1.0000001192092896, 6.931469440460205e-1, 2.4022120237350464e-1, 5.5507123470306396e-2,
              9.675543755292892e-3, 1.3276718091219664e-3], dtype=np.float32)


def fma32(a, b, c):
    # the product of two floats is exact in float64; one float64 rounding before the float32 one (<= 1 ulp of slack)
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def poly(f):
    p = np.full(f.shape, C[5], np.float32)
    for k in (4, 3, 2, 1, 0):
        p = fma32(p, f, np.full(f.shape, C[k], np.float32))
    return p


def exp2_poly(t):
    """s1_exp2_poly in numpy float32"""
    t = np.maximum(t.astype(np.float32), np.float32(-125.0))
    j = (t + np.float32(12582912.0)).astype(np.float32)
    n = (j - np.float32(12582912.0)).astype(np.float32)
    f = fma32(n, np.full(n.shape, -1.0, np.float32), t)
    p = poly(f)
    bits = p.view(np.uint32) + (j.view(np.uint32) << np.uint32(23))
    return bits.view(np.float32)


def test_exp2_poly_every_reduced_argument():
    worst = 0.0
    for sign in (1.0, -1.0):
        for e in range(-13, -1):                                 # binade [2^e, 2^(e+1)), top binade up to 0.5
            lo = np.float32(2.0 ** e).view(np.uint32)
            bits = np.arange(lo, lo + (1 << 23), dtype=np.uint32)
            f = bits.view(np.float32) * np.float32(sign)
            rel = np.abs(poly(f).astype(np.float64) / np.exp2(f.astype(np.float64)) - 1.0)
            worst = max(worst, float(rel.max()))
    f = np.float32(0.5) * np.array([-1.0, 1.0], np.float32)
    worst = max(worst, float(np.abs(poly(f) / np.exp2(f.astype(np.float64)) - 1).max()))
    tiny = (np.random.default_rng(0).uniform(-1, 1, 1 << 22) * 2.0 ** -12).astype(np.float32)
    tiny = np.concatenate([tiny, np.array([0.0, -0.0, 1e-45, -1e-45, 1e-30], np.float32)])
    worst = max(worst, float(np.abs(poly(tiny) / np.exp2(tiny.astype(np.float64)) - 1).max()))
    print(f"max relative error of the 2^f polynomial: {worst:.3g} ({np.log2(worst):.2f} bits)")
    assert worst <= 2.0 ** -21


def test_exp2_poly_exponent_and_clamp():
    rng = np.random.default_rng(1)
    t = np.concatenate([rng.uniform(-125, 0, 1 << 20), -np.arange(0, 125.5, 0.5), [-0.0, -124.9999]]).astype(np.float32)
    got = exp2_poly(t).astype(np.float64)
    rel = np.abs(got / np.exp2(t.astype(np.float64)) - 1)
    assert rel.max() <= 2.0 ** -21
    # below the clamp: a normal number at most 2^-124.5 (ex2.approx.ftz gives 0 or a subnormal there)
    low = exp2_poly(np.array([-126.0, -200.0, -1e30, -np.inf], np.float32)).astype(np.float64)
    assert np.all(low > 0) and np.all(low <= 2.0 ** -124.5) and np.all(low >= 2.0 ** -126)


def split16(v):
    hi = v.astype(np.float16).astype(np.float32)
    lo = (v - hi).astype(np.float16).astype(np.float32)
    return hi, lo


def paths(x, b, b2):
    """r^2 of every (candidate, training point): the full launch's FP32 chain, the split MMA path (FP32 accumulation
    in order: lo products from zero, then hi.hi with the norms), the exact value of the same FP32 inputs, and T"""
    d = x.shape[1]
    a2 = np.zeros(len(x), np.float32)
    for j in range(d):
        a2 = fma32(x[:, j], x[:, j], a2)
    a2 = (np.float32(0.25) * a2).astype(np.float32)
    A2, B2 = np.broadcast_arrays(a2[:, None], b2[None, :])
    rf = (A2 + B2).astype(np.float32)
    for j in range(d):
        rf = fma32(np.broadcast_to(x[:, j:j + 1], rf.shape), np.broadcast_to(b[None, :, j], rf.shape), rf)
    xh, xl = split16(x)
    bh, bl = split16(b)
    a2h, a2l = split16(a2)
    b2h, b2l = split16(b2)
    f64 = np.float64
    lo1 = (xl.astype(f64) @ bh.T.astype(f64)).astype(np.float32)
    lo2 = (lo1 + (xh.astype(f64) @ bl.T.astype(f64))).astype(np.float32)
    hh = xh.astype(f64) @ bh.T.astype(f64) + (a2h + a2l)[:, None].astype(f64) + (b2h + b2l)[None, :].astype(f64)
    rt = (lo2 + hh).astype(np.float32)
    exact = a2[:, None].astype(f64) + b2[None, :].astype(f64) + x.astype(f64) @ b.T.astype(f64)
    T = (np.sqrt(a2.astype(f64))[:, None] + np.sqrt(f64(b2.max()))) ** 2
    return a2, rf, rt, exact, T


def cases():
    rng = np.random.default_rng(7)
    for d, scale in ((10, 1.0), (1, 1.0), (12, 1.0), (10, 40.0), (6, 1e-4), (3, 300.0)):
        tr = (rng.random((256, d)) - 0.5) * scale                   # (X - c) / ell: training points
        cand = (rng.random((300, d)) - 0.5) * scale
        cand = np.concatenate([cand, tr[:40], tr[:10] + 1e-7 * scale])   # training rows as candidates
        b = tr.astype(np.float32)
        x = (-2.0 * cand).astype(np.float32)
        b2 = np.zeros(len(b), np.float32)
        for j in range(d):
            b2 = fma32(b[:, j], b[:, j], b2)
        yield d, scale, x, b, b2


@pytest.mark.parametrize("case", list(range(6)))
def test_distance_paths_within_the_r2_bounds(case):
    d, scale, x, b, b2 = list(cases())[case]
    _, rf, rt, exact, T = paths(x, b, b2)
    assert np.all(np.abs(rf - exact) <= G_F * U * T), (d, scale)
    assert np.all(np.abs(rt - exact) <= G_TC * U * T + E_SUB), (d, scale)


def k_matern_full(r2):                                       # gen8_kval: signed r^2 in the 5/3 r^2 term
    r = np.sqrt(np.abs(r2))
    return (1 + np.sqrt(5) * r + 5.0 / 3.0 * r2) * np.exp(-np.sqrt(5) * r)


def k_matern_tc(r2):                                         # s1_columns: the Matern function of r = sqrt|r^2|
    r = np.sqrt(np.abs(r2))
    return (1 + np.sqrt(5) * r + 5.0 / 3.0 * r * r) * np.exp(-np.sqrt(5) * r)


@pytest.mark.parametrize("case", list(range(6)))
@pytest.mark.parametrize("matern", [True, False])
def test_margin_covers_the_mean_difference(case, matern):
    d, scale, x, b, b2 = list(cases())[case]
    a2, rf, rt, _, T = paths(x, b, b2)
    c = np.random.default_rng(case).normal(0, 30, len(b)).astype(np.float32)
    kf = k_matern_full(rf.astype(np.float64)) if matern else np.exp(-0.5 * rf.astype(np.float64))
    kt = k_matern_tc(rt.astype(np.float64)) if matern else np.exp(-0.5 * rt.astype(np.float64))
    mu_f, mu_t, A = kf @ c, kt @ c, kt @ np.abs(c)
    S = float(np.abs(c).sum())
    e_f = G_F * U * T[:, 0]
    e_r = (G_F + G_TC) * U * T[:, 0] + E_SUB
    ok = e_r <= 0.0078125
    lr = (5 / 6) * 1.05 * e_r + (10 / 3) * 1.02 * e_f if matern else 0.5 * 1.05 * e_r
    zeta = (3.0 * 256 / 64 + 16) * U
    M = SAFETY * ((lr + ETA + zeta) * 1.05 * A + ETA_ABS * S)
    assert np.all(np.abs(mu_t - mu_f)[ok] <= M[ok]), (d, scale)
    worst = float((np.abs(mu_t - mu_f)[ok] / M[ok]).max()) if ok.any() else 0.0
    print(f"d {d} scale {scale}: max |mu~ - mu_F| / M = {worst:.3g}, {int((~ok).sum())} candidates without a bound")


def staircase(rng, p):
    f1 = np.sort(rng.random(p))[::-1]
    f2 = np.sort(rng.random(p))
    return np.column_stack([f1, f2]), np.array([1.2, 1.3])


@pytest.mark.parametrize("seed", range(6))
def test_exact_ehvi_non_increasing_in_mu(seed):
    rng = np.random.default_rng(seed)
    PF, r = staircase(rng, int(rng.integers(1, 40)))
    m = 300
    base = rng.uniform(-0.5, 1.8, (m, 2))
    var = rng.uniform(1e-4, 1.0, (m, 2))
    steps = np.linspace(-3.0, 3.0, 61)
    for obj in (0, 1):
        prev = None
        for s in steps:                                       # the mean of one objective grows
            mu = base.copy()
            mu[:, obj] += s
            v = O.ehvi_batched(mu[:, 0], mu[:, 1], var[:, 0], var[:, 1], PF, r, None, "exact")
            assert np.all(np.isfinite(v)) and np.all(v >= 0)
            if prev is not None:
                assert np.all(v <= prev + 1e-12 * np.abs(prev) + 1e-300), (obj, s)
            prev = v
