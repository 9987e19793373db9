"""Candidate-independent, once-per-iteration preparation ON THE DEVICE (SURVEY.md section 8f rank 2).

Device twins of `host_prep.calc_pf / pareto_mask / hypervolume / decompose_into_cells / ehvi_boxes`: the
reference gets these from pygmo (`fast_non_dominated_sorting` util_functions.py:76,
`hypervolume.compute` :198-199) and pymoo (`HV` optimisers.py:217-219) once per BO iteration;
they are O(n^2) on the evaluated samples and start to matter next to a ~100 ms scoring pass once
n reaches the thousands.  Results are bit-identical to the host versions (same comparison and
summation order, no FMA contraction), which the GPU tests assert.  Inputs may be numpy arrays or
torch tensors (copied to `device` as float64 if they are not there already)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _cabi
from .gp import _as_device, current_stream_ptr


def _dev_f64(a, device):
    t = a if torch.is_tensor(a) else torch.as_tensor(np.ascontiguousarray(np.asarray(a, dtype=np.float64)))
    t = t.to(device=device, dtype=torch.float64)
    return t.reshape(1, -1).contiguous() if t.ndim == 1 else t.contiguous()


def _vec(v, k):
    v = np.asarray(v.detach().cpu() if torch.is_tensor(v) else v, dtype=np.float64).reshape(-1)
    if len(v) != k:
        raise ValueError(f"expected {k} components, got {len(v)}")
    return (C.c_double * k)(*v)


def pareto_mask(Y, device="cuda:0"):
    """(n,) bool tensor on the device: True for the rows of Y (n,k) in the first non-dominated front."""
    dev = _as_device(device)
    Yd = _dev_f64(Y, dev)
    n, k = Yd.shape
    mask = torch.empty((n,), dtype=torch.uint8, device=dev)
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_pareto_mask(ctx.handle, C.c_void_p(Yd.data_ptr()), n, k,
                                                 C.c_void_p(mask.data_ptr()), current_stream_ptr(dev)))
    return mask.bool()


def calc_pf(Y, device="cuda:0"):
    """First non-dominated front in original row order as a numpy array; fewer than two rows are
    returned unchanged (util_functions.py:64-77)."""
    Yn = np.asarray(Y.detach().cpu() if torch.is_tensor(Y) else Y, dtype=np.float64)
    if len(Yn) < 2:
        return Yn
    return Yn[pareto_mask(Yn, device).cpu().numpy()]


def hypervolume(points, ref_point, device="cuda:0"):
    """Exact dominated hypervolume (minimisation) of (p,k) points, k = 2 or 3."""
    dev = _as_device(device)
    P = _dev_f64(points, dev)
    p, k = P.shape
    out = torch.zeros((1,), dtype=torch.float64, device=dev)
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_hypervolume(ctx.handle, C.c_void_p(P.data_ptr()), p, k, _vec(ref_point, k),
                                                 C.c_void_p(out.data_ptr()), current_stream_ptr(dev)))
    return float(out.item())


def decompose_into_cells(pf, ideal_point, max_point, device="cuda:0"):
    """(p+1, 2, 2) cells of a 2-D front ([c][0] upper, [c][1] lower corner) as a device tensor."""
    dev = _as_device(device)
    P = _dev_f64(pf, dev)
    if P.shape[1] != 2:
        raise ValueError("cell decomposition is 2-D only (emo.py:21)")
    p = P.shape[0]
    cells = torch.empty((p + 1, 2, 2), dtype=torch.float64, device=dev)
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().ombo_cells_2d(ctx.handle, C.c_void_p(P.data_ptr()), p, _vec(ideal_point, 2),
                                              _vec(max_point, 2), C.c_void_p(cells.data_ptr()),
                                              current_stream_ptr(dev)))
    return cells


_boxes_guess = {}     # device -> the box count of the last call, the first buffer size of the next


def ehvi_boxes(PF, ref_point, device="cuda:0"):
    """(table, boxes) of `host_prep.ehvi_boxes(PF, ref_point)` as device float64 tensors, equal to it element for
    element and in its order: table (k, B), boxes (n_boxes, 2, k) breakpoint indices.  2 <= k <= 4; at most 16384 rows
    and 512 distinct front points inside ref_point.  The box buffer starts at the size of the previous call on the
    device and is reallocated once when the decomposition needs more."""
    dev = _as_device(device)
    r = np.asarray(ref_point.detach().cpu() if torch.is_tensor(ref_point) else ref_point, dtype=np.float64).reshape(-1)
    k = len(r)
    if not 2 <= k <= 4:
        raise ValueError(f"ehvi_boxes takes 2 to 4 objectives (got {k})")
    if not np.all(np.isfinite(r)):
        raise ValueError(f"ehvi_boxes needs a finite reference point (got {r})")
    shape = tuple(PF.shape) if torch.is_tensor(PF) else np.shape(PF)
    size = int(np.prod(shape))
    if (len(shape) == 2 and shape[1] != k) or len(shape) > 2 or size % k:
        raise ValueError(f"PF must be (p, {k}) for a {k}-objective reference point (got shape {shape})")
    p = size // k
    if p > 16384:
        raise ValueError(f"ehvi_boxes takes at most 16384 rows (got {p})")
    P = _dev_f64(PF, dev).reshape(p, k) if p else torch.empty((0, k), dtype=torch.float64, device=dev)
    table = torch.empty((k * (p + 2),), dtype=torch.float64, device=dev)
    B, n_boxes = C.c_int(), C.c_int64()
    cap = _boxes_guess.get(dev.index, 4096)
    ctx = _cabi.Context.get(dev.index)
    with torch.cuda.device(dev):
        for attempt in range(2):
            boxes = torch.empty((cap * 2 * k,), dtype=torch.float64, device=dev)
            rc = _cabi.lib().ombo_ehvi_boxes(ctx.handle, C.c_void_p(P.data_ptr()), p, k, _vec(r, k),
                                             C.c_void_p(table.data_ptr()), C.c_void_p(boxes.data_ptr()), cap,
                                             C.byref(B), C.byref(n_boxes), current_stream_ptr(dev))
            if rc != _cabi.ERR_SPACE or attempt:
                break
            cap = int(n_boxes.value)
        _cabi.check(rc)
    n = int(n_boxes.value)
    _boxes_guess[dev.index] = n
    return table[: k * B.value].view(k, B.value), boxes[: n * 2 * k].view(n, 2, k)
