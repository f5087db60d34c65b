"""ctypes view of the C ABI in ``include/fccqp.h`` (``libfccqp_b200.so``).

The library is built in-tree by ``fcc_qp_b200.build`` / ``__graft_entry__.build()``.
There is no fallback: if the shared object is missing, importing the solver
classes raises, and if no CUDA device is usable every compute call fails with
``FCCQPError`` (``FCCQP_E_CUDA``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# FCCQP_LIB: developer override (e.g. an instrumented -DFCCQP_DEV build of the same sources)
LIB_PATH = os.environ.get("FCCQP_LIB") or os.path.join(_HERE, "libfccqp_b200.so")

ABI_VERSION = 5
STRUCTURE_AUTO, STRUCTURE_DENSE, STRUCTURE_CAPS = 0, 1, 2
STRUCTURE_REFINE = 256   # flag: iterative refinement of the reduced cold pre-solve
SCHEDULE_LPT = 512       # flag: n_iter holds an earlier solve's counts; lanes that ran long are processed first
MEM_HOST, MEM_DEVICE = 0, 1
STATUS_SUCCESS, STATUS_MAX_ITERATIONS, STATUS_NUMERICAL_ISSUE = 0, 1, 2
E_INVALID, E_CUDA, E_UNSUPPORTED = -1, -2, -3

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class FCCQPError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"fccqp error {code}: {msg}")
        self.code = code


class Options(C.Structure):
    _fields_ = [("max_iter", C.c_int32), ("adapt_rho_interval", C.c_int32), ("rho", C.c_double),
                ("eps_fcone", C.c_double), ("eps_bound", C.c_double), ("relaxation", C.c_double)]


class Details(C.Structure):
    _fields_ = [("n_iter", C.c_int32), ("solve_status", C.c_int32),
                ("admm_residual_bounds", C.c_double), ("admm_residual_friction_cone", C.c_double),
                ("solve_time", C.c_double), ("factorization_time", C.c_double),
                ("bounds_viol", C.c_double), ("friction_cone_viol", C.c_double)]


class BatchDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("batch", C.c_int32),
        ("n", C.c_int32), ("m", C.c_int32), ("nc", C.c_int32), ("lambda_c_start", C.c_int32),
        ("device", C.c_int32), ("memory_space", C.c_int32), ("precision", C.c_int32),
        ("warm_start", C.c_int32),
        ("options", Options),
        ("Q", C.c_void_p), ("q_batch_stride", C.c_int64), ("q_row_stride", C.c_int64), ("q_col_stride", C.c_int64),
        ("b", C.c_void_p), ("b_batch_stride", C.c_int64),
        ("A_eq", C.c_void_p), ("a_batch_stride", C.c_int64), ("a_row_stride", C.c_int64), ("a_col_stride", C.c_int64),
        ("b_eq", C.c_void_p), ("beq_batch_stride", C.c_int64),
        ("friction_coeffs", C.c_void_p), ("mu_batch_stride", C.c_int64),
        ("lb", C.c_void_p), ("lb_batch_stride", C.c_int64),
        ("ub", C.c_void_p), ("ub_batch_stride", C.c_int64),
        ("x", C.c_void_p), ("mu_x", C.c_void_p), ("mu_lambda_c", C.c_void_p),
        ("n_iter", C.c_void_p), ("status", C.c_void_p),
        ("res_bounds", C.c_void_p), ("res_fcone", C.c_void_p),
        ("bounds_viol", C.c_void_p), ("fcone_viol", C.c_void_p),
        ("stream", C.c_void_p),
        ("device_seconds", _dp),
        ("structure", C.c_int32), ("struct_caps", C.c_int32 * 3),
        ("warm_lanes", C.c_void_p),
    ]


class WbcDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("batch", C.c_int32),
        ("nv", C.c_int32), ("nu", C.c_int32), ("nh", C.c_int32), ("nc", C.c_int32), ("ny", C.c_int32),
        ("device", C.c_int32),
        ("w_vdot", C.c_double), ("w_u", C.c_double), ("w_lambda_c", C.c_double), ("w_eps", C.c_double),
        ("M", C.c_void_p), ("M_batch_stride", C.c_int64),
        ("Jh", C.c_void_p), ("Jh_batch_stride", C.c_int64),
        ("Jc", C.c_void_p), ("Jc_batch_stride", C.c_int64),
        ("Jy", C.c_void_p), ("Jy_batch_stride", C.c_int64),
        ("W", C.c_void_p), ("W_batch_stride", C.c_int64),
        ("ydd_cmd", C.c_void_p), ("ydd_batch_stride", C.c_int64),
        ("bias", C.c_void_p), ("bias_batch_stride", C.c_int64),
        ("gamma_h", C.c_void_p), ("gh_batch_stride", C.c_int64),
        ("gamma_c", C.c_void_p), ("gc_batch_stride", C.c_int64),
        ("Q", C.c_void_p), ("b", C.c_void_p), ("A_eq", C.c_void_p), ("b_eq", C.c_void_p),
        ("stream", C.c_void_p),
    ]


class PolishDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("batch", C.c_int32), ("n", C.c_int32), ("m", C.c_int32), ("nc", C.c_int32),
        ("lambda_c_start", C.c_int32), ("device", C.c_int32), ("reserved", C.c_int32),
        ("eps_fcone", C.c_double), ("eps_bound", C.c_double), ("eps_objective", C.c_double),
        ("Q", C.c_void_p), ("q_batch_stride", C.c_int64),
        ("b", C.c_void_p), ("b_batch_stride", C.c_int64),
        ("A_eq", C.c_void_p), ("a_batch_stride", C.c_int64),
        ("b_eq", C.c_void_p), ("beq_batch_stride", C.c_int64),
        ("friction_coeffs", C.c_void_p), ("mu_batch_stride", C.c_int64),
        ("lb", C.c_void_p), ("lb_batch_stride", C.c_int64),
        ("ub", C.c_void_p), ("ub_batch_stride", C.c_int64),
        ("x", C.c_void_p), ("mu_x", C.c_void_p), ("mu_lambda_c", C.c_void_p),
        ("Qp", C.c_void_p), ("bp", C.c_void_p), ("Ap", C.c_void_p), ("beqp", C.c_void_p),
        ("rot", C.c_void_p),
        ("y", C.c_void_p), ("y_status", C.c_void_p),
        ("z", C.c_void_p), ("bounds_viol", C.c_void_p), ("fcone_viol", C.c_void_p),
        ("polished", C.c_void_p),
        ("stream", C.c_void_p),
    ]


# every symbol include/fccqp.h declares (tests check that the library exports them all)
EXPORTS = [
    "fccqp_default_options", "fccqp_last_error", "fccqp_abi_version", "fccqp_device_count",
    "fccqp_create", "fccqp_destroy", "fccqp_set_options", "fccqp_get_options", "fccqp_set_rho",
    "fccqp_set_max_iter", "fccqp_set_warm_start", "fccqp_contact_vars_start", "fccqp_solve",
    "fccqp_get_solution", "fccqp_get_warm_state", "fccqp_set_warm_state", "fccqp_batch_solve",
    "fccqp_release_workspaces", "fccqp_kernel_launch_count", "fccqp_last_launch_info",
    "fccqp_alloc_pinned", "fccqp_free_pinned", "fccqp_wbc_assemble",
    "fccqp_last_struct_info", "fccqp_set_structure", "fccqp_batch_solve_multi", "fccqp_measure_fp64_peak",
    "fccqp_polish_prepare", "fccqp_polish_finish", "fccqp_batch_solve_rho", "fccqp_batch_solve_multi_rho",
]

_lib = None


def lib() -> C.CDLL:
    """Load libfccqp_b200.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m fcc_qp_b200.build` "
            "(needs nvcc; the solver has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.fccqp_last_error.restype = C.c_char_p
    L.fccqp_default_options.argtypes = [C.POINTER(Options)]
    L.fccqp_create.argtypes = [C.c_int] * 5 + [C.POINTER(C.c_void_p)]
    L.fccqp_destroy.argtypes = [C.c_void_p]
    L.fccqp_set_options.argtypes = [C.c_void_p, C.POINTER(Options)]
    L.fccqp_get_options.argtypes = [C.c_void_p, C.POINTER(Options)]
    L.fccqp_set_rho.argtypes = [C.c_void_p, C.c_double]
    L.fccqp_set_max_iter.argtypes = [C.c_void_p, C.c_int]
    L.fccqp_set_warm_start.argtypes = [C.c_void_p, C.c_int]
    L.fccqp_contact_vars_start.argtypes = [C.c_void_p]
    L.fccqp_solve.argtypes = [C.c_void_p, _dp, C.c_ssize_t, C.c_ssize_t, _dp, _dp, C.c_ssize_t,
                              C.c_ssize_t, _dp, _dp, C.c_int, _dp, _dp]
    L.fccqp_get_solution.argtypes = [C.c_void_p, _dp, C.POINTER(Details)]
    L.fccqp_get_warm_state.argtypes = [C.c_void_p, _dp, _dp, _dp]
    L.fccqp_set_warm_state.argtypes = [C.c_void_p, _dp, _dp, _dp]
    L.fccqp_batch_solve.argtypes = [C.POINTER(BatchDesc)]
    L.fccqp_batch_solve_multi.argtypes = [C.POINTER(BatchDesc), C.POINTER(C.c_int32), C.c_int32]
    L.fccqp_batch_solve_rho.argtypes = [C.POINTER(BatchDesc), C.c_void_p]
    L.fccqp_batch_solve_multi_rho.argtypes = [C.POINTER(BatchDesc), C.c_void_p, C.POINTER(C.c_int32), C.c_int32]
    L.fccqp_kernel_launch_count.restype = C.c_int64
    L.fccqp_measure_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.fccqp_last_launch_info.argtypes = [_ip, _ip, _ip, _ip]
    L.fccqp_last_struct_info.argtypes = [_ip, _ip, _ip, _ip, _ip]
    L.fccqp_set_structure.argtypes = [C.c_void_p, C.c_int]
    L.fccqp_alloc_pinned.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    L.fccqp_free_pinned.argtypes = [C.c_void_p]
    L.fccqp_wbc_assemble.argtypes = [C.POINTER(WbcDesc)]
    L.fccqp_polish_prepare.argtypes = [C.POINTER(PolishDesc)]
    L.fccqp_polish_finish.argtypes = [C.POINTER(PolishDesc)]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise FCCQPError(rc, lib().fccqp_last_error().decode())


def last_launch_info() -> dict:
    g, b, s, c = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    lib().fccqp_last_launch_info(C.byref(g), C.byref(b), C.byref(s), C.byref(c))
    return dict(grid=g.value, block=b.value, smem_bytes=s.value, ctas_per_sm=c.value)


def last_struct_info() -> dict:
    """What the last batch launch did about problem structure (``fccqp_last_struct_info``); ``deferred`` is
    valid once the stream of that call has been synchronised."""
    used, rows, dense, deferred = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    caps = (C.c_int32 * 3)()
    lib().fccqp_last_struct_info(C.byref(used), caps, C.byref(rows), C.byref(dense), C.byref(deferred))
    return dict(used=bool(used.value), caps=tuple(int(c) for c in caps), rows=rows.value, rows_dense=dense.value,
                deferred=deferred.value)


def pinned_empty(shape, dtype):
    """numpy array in page-locked host memory (``fccqp_alloc_pinned``): the batched host path
    moves such arrays by asynchronous DMA.  Freed when the array (and its views) are collected."""
    import weakref

    import numpy as np
    dtype = np.dtype(dtype)
    count = int(np.prod(shape, dtype=np.int64))
    nbytes = max(count * dtype.itemsize, 1)
    ptr = C.c_void_p()
    check(lib().fccqp_alloc_pinned(nbytes, C.byref(ptr)))
    buf = (C.c_char * nbytes).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)
    weakref.finalize(buf, lib().fccqp_free_pinned, ptr.value)
    return arr
