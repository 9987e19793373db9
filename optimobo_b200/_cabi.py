"""ctypes binding of the C ABI declared in include/optimobo_b200.h.

There is NO fallback: if the shared library is missing or a call fails, an exception is raised.
The library is built in-tree by `__graft_entry__.build()` / `make -C optimobo_b200/csrc`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liboptimobo_b200.so")

OK, ERR_INVALID, ERR_NOT_PD, ERR_CUDA, ERR_UNSUPPORTED = 0, -1, -2, -3, -4
MAX_GP, MAX_OBJ, MAX_DIM, MAX_TRAIN = 8, 4, 32, 8192

KERNEL_MATERN52, KERNEL_RBF = 0, 1
PREC_FP64, PREC_FAST = 0, 1
SEM_REFERENCE, SEM_EXACT = 0, 1
(ACQ_NONE, ACQ_EHVI2D, ACQ_EHVI3D, ACQ_EXPECTED_DECOMP, ACQ_EI, ACQ_CONSTRAINED_EI,
 ACQ_PARETO_EI, ACQ_HV_POI) = range(8)
ACQ_EHVI_BOX = 8
EHVI_BOX_MAX_BREAKS, EHVI_BOX_MAX_BOXES = 514, 1 << 20
(FIELD_L, FIELD_LINV, FIELD_ALPHA, FIELD_XS, FIELD_STATUS, FIELD_BHI, FIELD_BLO, FIELD_XS32,
 FIELD_ALPHA32) = range(9)

EXPORTS = [
    "ombo_abi_version", "ombo_has_fast_path", "ombo_last_error", "ombo_ctx_create", "ombo_ctx_destroy", "ombo_n_pad",
    "ombo_gp_state_bytes", "ombo_gp_state_field", "ombo_gp_refresh", "ombo_gp_nlml_grad", "ombo_score",
    "ombo_score_host", "ombo_acquire_posterior", "ombo_pool_rows", "ombo_launch_count",
    "ombo_pack_key", "ombo_profile_enable", "ombo_profile_read",
    "ombo_pareto_mask", "ombo_hypervolume", "ombo_cells_2d", "ombo_posterior_joint_samples", "ombo_scalarise",
]


class GpSpec(C.Structure):
    _fields_ = [("n", C.c_int32), ("d", C.c_int32), ("kernel", C.c_int32), ("reserved", C.c_int32),
                ("sigma_f2", C.c_double), ("sigma_n2", C.c_double), ("jitter", C.c_double),
                ("X", C.c_void_p), ("y", C.c_void_p), ("ell", C.POINTER(C.c_double))]


class Gp(C.Structure):
    _fields_ = [("n", C.c_int32), ("d", C.c_int32), ("kernel", C.c_int32), ("reserved", C.c_int32),
                ("sigma_f2", C.c_double), ("sigma_n2", C.c_double), ("var_floor", C.c_double),
                ("state", C.c_void_p)]


class Pool(C.Structure):
    _fields_ = [("X", C.c_void_p), ("dtype", C.c_int32), ("d", C.c_int32), ("m", C.c_int64),
                ("index_base", C.c_int64), ("seed", C.c_uint64),
                ("lo", C.c_double * MAX_DIM), ("hi", C.c_double * MAX_DIM)]


class Acq(C.Structure):
    _fields_ = [("kind", C.c_int32), ("semantics", C.c_int32), ("scalarisation", C.c_int32),
                ("n_obj", C.c_int32), ("n_pf", C.c_int32), ("n_cells", C.c_int32),
                ("n_samples", C.c_int32), ("reserved", C.c_int32),
                ("best", C.c_double), ("var_eps", C.c_double * MAX_GP),
                ("ref", C.c_double * MAX_OBJ), ("ideal", C.c_double * MAX_OBJ),
                ("maxp", C.c_double * MAX_OBJ), ("weights", C.c_double * MAX_OBJ),
                ("sc_params", C.c_double * 4), ("cache_c00", C.c_double), ("cache_c01", C.c_double),
                ("stripes", C.c_void_p), ("cells", C.c_void_p), ("cache", C.c_void_p)]


class Best(C.Structure):
    _fields_ = [("value", C.c_double), ("index", C.c_int64)]


class OmboError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"optimobo_b200 C ABI error {code}: {msg}")
        self.code = code


class NotPositiveDefinite(OmboError):
    pass


_lib = None


def lib():
    """Loads liboptimobo_b200.so (once).  Fails loudly -- there is no CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()' or make -C optimobo_b200/csrc). "
            "optimobo_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    L.ombo_abi_version.restype = C.c_int
    L.ombo_last_error.restype = C.c_char_p
    L.ombo_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.ombo_ctx_destroy.argtypes = [C.c_void_p]
    L.ombo_n_pad.argtypes = [C.c_int]
    L.ombo_gp_state_bytes.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_size_t)]
    L.ombo_gp_state_field.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.ombo_gp_refresh.argtypes = [C.c_void_p, C.POINTER(GpSpec), C.c_void_p, C.c_void_p]
    L.ombo_gp_nlml_grad.argtypes = [C.c_void_p, C.POINTER(GpSpec), C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
    L.ombo_score.argtypes = [C.c_void_p, C.POINTER(Gp), C.c_int, C.POINTER(Pool), C.POINTER(Acq), C.c_int,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ombo_score_host.argtypes = [C.c_void_p, C.POINTER(Gp), C.c_int, C.POINTER(Pool), C.POINTER(Acq),
                                  C.c_int, C.POINTER(Best), C.c_void_p]
    L.ombo_acquire_posterior.argtypes = [C.c_void_p, C.POINTER(Acq), C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                         C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ombo_scalarise.argtypes = [C.c_void_p, C.POINTER(Acq), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.ombo_pool_rows.argtypes = [C.c_void_p, C.POINTER(Pool), C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
    L.ombo_pack_key.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ombo_pareto_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.ombo_hypervolume.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_void_p,
                                   C.c_void_p]
    L.ombo_cells_2d.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                C.c_void_p, C.c_void_p]
    L.ombo_posterior_joint_samples.argtypes = [C.c_void_p, C.POINTER(Gp), C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                               C.c_double, C.c_void_p, C.c_void_p]
    L.ombo_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.ombo_profile_read.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    L.ombo_launch_count.argtypes = [C.c_void_p, C.c_int]
    L.ombo_launch_count.restype = C.c_int64
    for name in EXPORTS:
        getattr(L, name)
    _lib = L
    return L


def fast_path_available() -> bool:
    return bool(lib().ombo_has_fast_path())


def check(rc):
    if rc == OK:
        return
    msg = lib().ombo_last_error().decode("utf-8", "replace")
    if rc == ERR_NOT_PD:
        raise NotPositiveDefinite(rc, msg)
    raise OmboError(rc, msg)


def state_bytes(n, d):
    b = C.c_size_t()
    check(lib().ombo_gp_state_bytes(n, d, C.byref(b)))
    return b.value


def state_field(n, d, field):
    off, cnt = C.c_size_t(), C.c_size_t()
    check(lib().ombo_gp_state_field(n, d, field, C.byref(off), C.byref(cnt)))
    return off.value, cnt.value


class Context:
    """One per device (and per thread using it)."""

    _by_device = {}

    def __init__(self, device: int):
        self.device = int(device)
        h = C.c_void_p()
        check(lib().ombo_ctx_create(self.device, C.byref(h)))
        self.handle = h

    @classmethod
    def get(cls, device: int) -> "Context":
        device = int(device)
        if device not in cls._by_device:
            cls._by_device[device] = Context(device)
        return cls._by_device[device]

    def launch_count(self, reset=False) -> int:
        return int(lib().ombo_launch_count(self.handle, 1 if reset else 0))

    def profile(self, enable=True):
        check(lib().ombo_profile_enable(self.handle, 1 if enable else 0))

    def profile_read(self):
        n, ms = C.c_int64(), C.c_double()
        check(lib().ombo_profile_read(self.handle, C.byref(n), C.byref(ms)))
        return int(n.value), float(ms.value)

    def close(self):
        if self.handle:
            lib().ombo_ctx_destroy(self.handle)
            self.handle = None
            Context._by_device.pop(self.device, None)
