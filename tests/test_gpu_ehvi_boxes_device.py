"""GPU: the box decomposition built on the device (ombo_ehvi_boxes, device_prep.ehvi_boxes) against its definition,
host_prep.ehvi_boxes -- equal arrays element for element and in order -- and the scores and optimiser runs built on
it against the host-built ones, bit for bit."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import optimobo_b200 as ob  # noqa: E402
from optimobo_b200 import _cabi, device_prep, host_prep  # noqa: E402
from optimobo_b200.algorithms import MultiSurrogateOptimiser  # noqa: E402
from optimobo_b200.gp import current_stream_ptr  # noqa: E402
from optimobo_b200.problem import Problem  # noqa: E402

DEV = "cuda:0"
needs_fast = pytest.mark.skipif(not _cabi.fast_path_available(), reason="fast path not built")


def _sphere(P, k, rng):
    X = np.abs(rng.normal(size=(P, k)))
    return X / np.linalg.norm(X, axis=1, keepdims=True)


def _antichain(P, k, rng):
    """Objectives 1, 2 a 2-D anti-chain and the rest one shared order: every subset is its own front, so the number
    of boxes grows as P^(k-1)."""
    t, z = rng.permutation(P) / P, rng.permutation(P) / P
    return np.column_stack([t, 1 - t] + [z] * (k - 2))


def _same(Y, r):
    table, boxes = host_prep.ehvi_boxes(Y, r)
    t_dev, b_dev = device_prep.ehvi_boxes(Y, r, DEV)
    assert t_dev.dtype == b_dev.dtype == torch.float64 and t_dev.device.type == b_dev.device.type == "cuda"
    t_dev, b_dev = t_dev.cpu().numpy(), b_dev.cpu().numpy()
    assert t_dev.shape == table.shape and b_dev.shape == boxes.shape, (t_dev.shape, table.shape, b_dev.shape,
                                                                        boxes.shape)
    assert np.array_equal(t_dev, table)
    assert np.array_equal(b_dev, boxes.astype(np.float64))
    return len(boxes)


@pytest.mark.parametrize("k", [2, 3, 4])
def test_tiny_fronts(k):
    r = np.full(k, 1.0)
    assert _same(np.empty((0, k)), r) == 1
    assert _same([], r) == 1
    _same(np.full((1, k), 0.5), r)
    _same(np.array([[0.2] * k, [0.5] * k]), r)                              # the second is dominated
    _same(np.array([[0.2] + [0.6] * (k - 1), [0.6] + [0.2] * (k - 1)]), r)
    _same(np.full((1, k), 1.0), r)                                          # a point at r itself
    _same(np.full((2, k), 2.0), r)                                          # nothing inside r


@pytest.mark.parametrize("k,P", [(2, 64), (2, 512), (3, 66), (3, 256), (3, 512), (4, 60), (4, 150), (4, 256)])
def test_sphere_fronts(k, P):
    rng = np.random.default_rng(10 * k + P)
    _same(_sphere(P, k, rng), np.full(k, 1.1))


@pytest.mark.parametrize("k,P", [(3, 512), (4, 90)])
def test_antichain_fronts(k, P):
    assert _same(_antichain(P, k, np.random.default_rng(P)), np.full(k, 1.1)) > P ** (k - 1) / 10


@pytest.mark.parametrize("k", [2, 3, 4])
def test_dominated_duplicate_nan_and_beyond_r_rows(k):
    rng = np.random.default_rng(k)
    F = _sphere(40, k, rng)
    Y = np.vstack([F, F[:7], F[:5] + 0.3, np.full((2, k), np.nan), F[:3] + 5.0, np.full((3, k), np.inf)])
    Y[-10, 0] = np.nan                                                       # one NaN coordinate in a front-like row
    Y = Y[rng.permutation(len(Y))]
    _same(Y, np.full(k, 1.1))
    _same(Y, np.full(k, 0.8))                                                # r cuts through the front


@pytest.mark.parametrize("k,P,levels", [(2, 200, 6), (3, 300, 5), (3, 300, 12), (4, 300, 5), (4, 400, 8)])
def test_integer_grid_ties_and_coordinates_at_r(k, P, levels):
    rng = np.random.default_rng(P + levels)
    Y = rng.integers(0, levels, size=(P, k)).astype(float)
    n = _same(Y, np.full(k, levels - 1.0))                                   # many coordinates equal r_i
    assert n >= 1
    _same(Y, np.full(k, levels - 2.0))
    _same(Y, np.arange(k) + levels / 2.0)


def test_whole_front_of_512_and_one_more():
    k = 3
    rng = np.random.default_rng(5)
    F = _sphere(513, k, rng)
    _same(F[:512], np.full(k, 1.1))
    _same(np.vstack([F[:512], F[:512]]), np.full(k, 1.1))                    # 1024 rows, 512 distinct
    with pytest.raises(_cabi.OmboError) as e:
        device_prep.ehvi_boxes(F, np.full(k, 1.1), DEV)
    assert e.value.code == _cabi.ERR_UNSUPPORTED and "513" in str(e.value)


def _raw(PF, r, cap):
    """ombo_ehvi_boxes itself: (rc, B, n_boxes, table, boxes)."""
    P = torch.as_tensor(np.asarray(PF, dtype=np.float64), device=DEV).contiguous()
    p, k = P.shape
    table = torch.full((k * (p + 2),), -7.0, dtype=torch.float64, device=DEV)
    boxes = torch.full((max(cap, 1) * 2 * k,), -7.0, dtype=torch.float64, device=DEV)
    B, nb = C.c_int(-1), C.c_int64(-1)
    ctx = _cabi.Context.get(0)
    rc = _cabi.lib().ombo_ehvi_boxes(ctx.handle, C.c_void_p(P.data_ptr()), p, k, (C.c_double * k)(*r),
                                     C.c_void_p(table.data_ptr()), C.c_void_p(boxes.data_ptr()), cap, C.byref(B),
                                     C.byref(nb), current_stream_ptr(torch.device(DEV)))
    torch.cuda.synchronize()
    return rc, B.value, nb.value, table.cpu().numpy(), boxes.cpu().numpy()


def test_space_status_and_retry():
    rng = np.random.default_rng(3)
    F, r = _sphere(100, 3, rng), [1.1] * 3
    table, boxes = host_prep.ehvi_boxes(F, r)
    rc, B, nb, t, b = _raw(F, r, 10)
    assert rc == _cabi.ERR_SPACE and (B, nb) == (table.shape[1], len(boxes))
    assert np.all(t == -7.0) and np.all(b == -7.0)                          # nothing written
    rc, B, nb, t, b = _raw(F, r, nb)
    assert rc == _cabi.OK
    assert np.array_equal(t[:3 * B].reshape(3, B), table) and np.array_equal(b.reshape(-1, 2, 3), boxes)
    # the wrapper starts from the last size and retries once
    device_prep._boxes_guess[0] = 1
    _same(F, r)
    assert device_prep._boxes_guess[0] == len(boxes)
    _same(_sphere(200, 3, rng), r)                                           # larger than the guess: one retry


def test_error_statuses():
    r = [1.0, 1.0, 1.0]
    with pytest.raises(_cabi.OmboError) as e:                                # -inf in a row inside r
        device_prep.ehvi_boxes([[0.5, 0.5, 0.5], [-np.inf, 0.9, 0.9]], r, DEV)
    assert e.value.code == _cabi.ERR_INVALID and "-inf" in str(e.value)
    device_prep.ehvi_boxes([[0.5, 0.5, 0.5], [-np.inf, 0.9, 2.0]], r, DEV)   # ... but not in a row beyond r
    # more boxes than the box EHVI takes (and ombo_score would reject)
    F = _antichain(200, 4, np.random.default_rng(8))
    with pytest.raises(_cabi.OmboError) as e:
        device_prep.ehvi_boxes(F, [1.1] * 4, DEV)
    assert e.value.code == _cabi.ERR_INVALID and "boxes" in str(e.value)
    rc, B, nb, _, _ = _raw(F, [1.1] * 4, 1 << 21)
    assert rc == _cabi.ERR_INVALID and nb > _cabi.EHVI_BOX_MAX_BOXES and B == 202
    # argument checks of the C entry
    for args in ((np.ones((2, 5)) * 0.5, [1.0] * 5), (np.ones((2, 1)) * 0.5, [1.0])):
        P = torch.as_tensor(args[0], device=DEV)
        rc = _cabi.lib().ombo_ehvi_boxes(_cabi.Context.get(0).handle, C.c_void_p(P.data_ptr()), 2, P.shape[1],
                                         (C.c_double * 5)(*([1.0] * 5)), C.c_void_p(P.data_ptr()),
                                         C.c_void_p(P.data_ptr()), 0, C.byref(C.c_int()), C.byref(C.c_int64()),
                                         None)
        assert rc == _cabi.ERR_INVALID
    rc = _cabi.lib().ombo_ehvi_boxes(_cabi.Context.get(0).handle, None, 0, 3, (C.c_double * 3)(1.0, np.nan, 1.0),
                                     C.c_void_p(P.data_ptr()), None, 0, C.byref(C.c_int()), C.byref(C.c_int64()), None)
    assert rc == _cabi.ERR_INVALID
    rc = _cabi.lib().ombo_ehvi_boxes(_cabi.Context.get(0).handle, C.c_void_p(P.data_ptr()), 16385, 2,
                                     (C.c_double * 2)(1.0, 1.0), C.c_void_p(P.data_ptr()), None, 0,
                                     C.byref(C.c_int()), C.byref(C.c_int64()), None)
    assert rc == _cabi.ERR_INVALID


# ------------------------------------------------------------------------------------------
# scoring with a device-built spec
# ------------------------------------------------------------------------------------------
def _models(k, c, rng, n=60, d=4):
    X = rng.random((n, d))
    cols = [np.sin(3 * X @ rng.normal(size=d)) for _ in range(k + c)]
    return [ob.GPModel(X, y, 0.6 * np.ones(d), 1.0, device=DEV) for y in cols]


@pytest.mark.parametrize("precision", ["fp64", pytest.param("fast", marks=needs_fast)])
@pytest.mark.parametrize("feasible", [False, True])
def test_score_bit_identical(precision, feasible):
    k, c = 3, 2
    rng = np.random.default_rng(11)
    models = _models(k, c if feasible else 0, rng)
    pool = ob.CandidatePool.counter(1 << 16, np.zeros(4), np.ones(4), seed=3)
    PF = np.vstack([_sphere(120, k, rng) * 0.8, _sphere(10, k, rng) + 0.5])
    r = np.full(k, 1.0)
    if feasible:
        host, dev = ob.spec_ehvi_box_feasible(r, PF, c), ob.spec_ehvi_box_feasible(r, PF, c, device=DEV)
    else:
        host, dev = ob.spec_ehvi_box(r, PF), ob.spec_ehvi_box(r, PF, device=DEV)
    assert torch.is_tensor(dev.stripes) and torch.is_tensor(dev.cells) and not torch.is_tensor(host.stripes)
    a = dev.c_struct(torch.device(DEV))
    assert a.stripes == dev.stripes.data_ptr() and a.cells == dev.cells.data_ptr()    # passed through, not copied
    assert (a.n_pf, a.n_cells) == (host.stripes.shape[1], host.cells.shape[0])
    h = ob.score(models, host, pool, precision=precision, want_acq=True)
    d = ob.score(models, dev, pool, precision=precision, want_acq=True)
    assert np.array_equal(h.acq.cpu().numpy(), d.acq.cpu().numpy())
    assert h.best_index == d.best_index and h.best_value == d.best_value


# ------------------------------------------------------------------------------------------
# the optimiser: the same run with the decomposition on the device and on the host
# ------------------------------------------------------------------------------------------
class DTLZ2(Problem):
    def __init__(self, n_obj=3, n_var=5, n_ieq_constr=0):
        super().__init__(n_var=n_var, n_obj=n_obj, n_ieq_constr=n_ieq_constr, vtype=float)
        self.xl, self.xu = np.zeros(n_var), np.ones(n_var)

    def _evaluate(self, x, out, *args, **kwargs):
        g = ((x[:, 2:] - 0.5) ** 2).sum(1)
        a, b = 0.5 * np.pi * x[:, 0], 0.5 * np.pi * x[:, 1]
        out["F"] = [(1 + g) * np.cos(a) * np.cos(b), (1 + g) * np.cos(a) * np.sin(b), (1 + g) * np.sin(a)]

    def _evaluate_constraints(self, x, out, *args, **kwargs):
        out["G"] = [x[:, 0] + x[:, 1] - 1.4]


class _Counting(MultiSurrogateOptimiser):
    def _box_device(self, front):
        dev = super()._box_device(front)
        self.on_device = getattr(self, "on_device", 0) + (dev is not None)
        return dev


@pytest.mark.parametrize("batch_size,constrained", [(1, False), (3, False), (1, True), (3, True)])
def test_optimiser_same_run(batch_size, constrained):
    problem = DTLZ2(n_ieq_constr=1 if constrained else 0)
    kw = dict(ehvi="box", constrained=constrained, batch_size=batch_size, n_candidates=1 << 14, seed=0, device=DEV,
              hyperparameters=(0.5 * np.ones(5), 1.0), refine_rounds=0)
    dev = _Counting(problem, [0, 0, 0], [2.5, 2.5, 2.5], prep_on_device=True, **kw)
    host = _Counting(problem, [0, 0, 0], [2.5, 2.5, 2.5], prep_on_device=False, **kw)
    a = dev.solve(budget=6, n_init_samples=20)
    b = host.solve(budget=6, n_init_samples=20)
    assert dev.on_device >= (6 if batch_size == 1 else 2) and host.on_device == 0
    np.testing.assert_array_equal(a.Xsample, b.Xsample)
    np.testing.assert_array_equal(a.hypervolume_convergence, b.hypervolume_convergence)
