"""Batched solver: B independent WBC QPs of identical dimensions per launch.

``FCCQPBatch`` mirrors the reference's ``FCCQP`` object (``src/fcc_qp.hpp:54-171``,
bound in ``src/main.cpp:42-54``) -- same constructor arguments, same
``set_options / set_rho / set_max_iter / set_warm_start / Solve / GetSolution``
method names and argument meaning -- but every problem argument carries a
leading batch dimension, and the carried warm-start state ``(x, mu_x,
mu_lambda_c)`` is a set of ``[B, .]`` arrays owned by the object.

Inputs are either numpy arrays (host memory; the C ABI stages them through the
GPU) or torch CUDA tensors / anything exposing ``__cuda_array_interface__`` via
``torch.as_tensor`` (device memory; zero-copy, asynchronous on the current torch
stream).  There is no CPU solve path.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import Any, Optional

import numpy as np

from . import _native as nat


@dataclasses.dataclass
class FCCQPOptionsB:
    """FCCQPOptions (``src/fcc_qp.hpp:30-35``) -- same fields and defaults."""
    max_iter: int = 1000
    rho: float = 1e-6
    eps_fcone: float = 1e-3
    eps_bound: float = 1e-6
    relaxation: float = 1.0   # extension (not in the reference): ADMM over-relaxation alpha in (0, 2); 1.0 = reference
    adapt_rho_interval: int = 0   # extension (not in the reference): adaptive rho every so many iterations; 0 = off


@dataclasses.dataclass
class BatchDetails:
    """FCCQPDetails (``src/fcc_qp.hpp:19-28``) as struct-of-arrays, python names of ``src/main.cpp:22-29``."""
    n_iter: Any
    eps_bounds: Any
    eps_friction_cone: Any
    bounds_viol: Any
    friction_cone_viol: Any
    solve_status: Any
    solve_time: float = 0.0          # host wall seconds of the whole batched call
    device_time: float = 0.0         # CUDA-event seconds of the solve kernel (device inputs) or staged call
    polished: Any = None             # after Polish(): 1 where the polished point replaced the ADMM one, 0 where it was rejected


@dataclasses.dataclass
class BatchSolution:
    """FCCQPSolution (``src/fcc_qp.hpp:37-40``): ``z`` is ``[B, n]``."""
    details: BatchDetails
    z: Any


def _is_torch(a) -> bool:
    return type(a).__module__.split(".")[0] == "torch"


class FCCQPBatch:
    def __init__(self, num_vars: int, num_equality_constraints: int, nc: int, lambda_c_start: int,
                 device=0, precision: str = "fp64"):
        if nc % 3 != 0:
            raise ValueError("nc must be a multiple of 3 (src/fcc_qp.cpp:32)")
        if lambda_c_start < 0 or lambda_c_start + nc > num_vars:
            raise ValueError("lambda_c_start + nc must be <= num_vars (src/fcc_qp.cpp:33)")
        self.n, self.m, self.nc, self.lcs = int(num_vars), int(num_equality_constraints), int(nc), int(lambda_c_start)
        # device: one CUDA ordinal, or a sequence of them -- host (numpy) batches are then split into contiguous shards,
        # one per device, inside ONE call (fccqp_batch_solve_multi: a host thread, streams and staging buffers per device)
        if isinstance(device, (list, tuple)):
            self.devices = [int(v) for v in device]
            if not self.devices:
                raise ValueError("device list is empty")
            self.device = self.devices[0]
        else:
            self.devices = None
            self.device = int(device)
        # "fp64": the reference's arithmetic and data.  "fp32_data": Q, b, A_eq, b_eq, friction_coeffs, lb, ub
        # travel and are stored as float32 (half the PCIe / HBM bytes), arithmetic, state and outputs stay
        # FP64 (FCCQP_PRECISION_FP32_DATA in include/fccqp.h; stated bound 2e-3 relative on z).  "fp32": float32 data AND FP32
        # arithmetic for problems with n + m <= 32 (the warp-per-QP kernel; FCCQP_PRECISION_FP32, stated bound 1e-3 relative
        # on z at cond <= 1e4 and eps >= 1e-4); larger problems run as "fp32_data".
        if precision not in ("fp64", "fp32_data", "fp32"):
            raise ValueError("precision must be 'fp64', 'fp32_data' or 'fp32'")
        self.precision = precision
        self.options = FCCQPOptionsB()
        # Problem structure (include/fccqp.h, fccqp_structure): "auto" sizes the structure-exploiting kernel from a
        # probe of the batch -- for device tensors on the first Solve() only (one stream synchronisation), the
        # bounds found are reused afterwards (QPs beyond them still run, on the general kernel, and the probe is
        # repeated when many do); "probe" probes on every call; "dense" never reduces; a 3-tuple gives the bounds.
        self.structure = "auto"
        # one step of iterative refinement of the reduced cold pre-solve (FCCQP_STRUCTURE_REFINE): 7e-11 instead of
        # 1.2e-7 relative on z against the reference on the walking log, ~25 % more time per cold QP
        self.refine = False
        # device (torch) path: lanes that ran long in the PREVIOUS Solve of this object are pulled from the work queue
        # first (FCCQP_SCHEDULE_LPT; the previous iteration counts are still in the solver-owned n_iter tensor).  For
        # control loops re-solving a slowly changing batch: the few QPs that run to max_iter stop being the tail of
        # the launch.  Changes the processing order only, never a result.
        self.schedule_from_previous = False
        self._caps = None
        self.warm_start = False
        self.warm_lanes = None  # per-lane mask of set_warm_start (None: warm_start holds for every lane)
        self.rho_lanes = None   # per-lane rho of set_rho, read and written by every Solve (None: options.rho for every lane)
        self.time_kernel = True
        self._state = None     # (x, mu_x, mu_c) arrays / tensors
        self._host_out = None  # page-locked output buffers of the numpy path
        self._dev_out = None   # device output / state tensors of the torch path
        self.zero_copy_outputs = False  # numpy path: GetSolution() returns views of those buffers
        self._sol: Optional[BatchSolution] = None
        nat.lib()              # fail loudly if the CUDA library is not built

    # --- same setters as the reference object (src/fcc_qp.hpp:75-91)
    def set_rho(self, rho):
        """A float: one rho for every lane, as on the reference object (clears a per-lane array).  Or a per-lane ``[B]``
        float64 array: lane i is solved as a reference object after ``set_rho(rho[i])``, and every ``Solve`` overwrites
        rho[i] with the rho lane i ended with -- under adaptive rho the next warm ``Solve`` continues from it, with the
        carried duals scaled for it (fccqp_batch_solve_rho in include/fccqp.h).  A numpy array for numpy batches, a
        contiguous CUDA tensor on the batch's device for device batches: kept, not copied, and read and written in place,
        so a captured CUDA graph carries it from replay to replay.  Entries of a device tensor that are not finite or
        not > 0 end their lane with status NUMERICAL_ISSUE and n_iter 0."""
        if _is_torch(rho):
            import torch
            if rho.dtype != torch.float64 or rho.dim() != 1:
                raise ValueError("a per-lane rho must be a 1-D float64 tensor")
            if rho.device.type != "cuda":
                raise ValueError("a torch per-lane rho must be a CUDA tensor (numpy arrays go with numpy batches)")
            if rho.numel() > 1 and rho.stride(0) != 1:
                raise ValueError("a per-lane rho must be contiguous (it is read and written in place)")
            self.rho_lanes = rho
        elif isinstance(rho, np.ndarray) and rho.ndim > 0:
            if rho.dtype != np.float64 or rho.ndim != 1:
                raise ValueError("a per-lane rho must be a 1-D float64 array")
            if not rho.flags.c_contiguous or not rho.flags.writeable:
                raise ValueError("a per-lane rho must be a contiguous, writeable array (it is written in place)")
            self._check_rho_values(rho)
            self.rho_lanes = rho
        else:
            if not rho > 0:
                raise ValueError("rho must be > 0")
            self.options.rho = float(rho)
            self.rho_lanes = None

    @staticmethod
    def _check_rho_values(rho: np.ndarray):
        if not np.all(np.isfinite(rho) & (rho > 0)):
            raise ValueError("every per-lane rho must be finite and > 0")

    def _rho_ptr(self, B: int, dev) -> int:
        """Pointer of the per-lane rho for a batch of B lanes (0: none); refuses an array that does not fit the call."""
        r = self.rho_lanes
        if r is None:
            return 0
        if r.shape[0] != B:
            raise ValueError(f"per-lane rho has {r.shape[0]} lanes, the batch {B}")
        if dev is None:
            if _is_torch(r):
                raise ValueError("numpy batch with a torch per-lane rho: pass a numpy array")
            self._check_rho_values(r)
            return r.ctypes.data
        if not _is_torch(r) or r.device != dev:
            raise ValueError(f"device batch on {dev} needs a CUDA per-lane rho on the same device")
        return r.data_ptr()

    def set_max_iter(self, n: int):
        if not n > 0:
            raise ValueError("max_iter must be > 0")
        self.options.max_iter = int(n)

    def set_options(self, opt):
        self.options = FCCQPOptionsB(int(opt.max_iter), float(opt.rho), float(opt.eps_fcone), float(opt.eps_bound),
                                     float(getattr(opt, "relaxation", 1.0)), int(getattr(opt, "adapt_rho_interval", 0)))

    def set_warm_start(self, warm_start):
        """``True`` / ``False`` for every lane, as on the reference object; or a per-lane ``[B]`` mask: lane i is solved
        as a reference object after ``set_warm_start(mask[i] != 0)`` -- warm from its carried state, or cold (pre-solve,
        zero duals).  A numpy bool / uint8 array for numpy batches (staged with the batch), a torch CUDA bool / uint8
        tensor for device batches: passed by pointer, read by the kernels when they run, so a mask updated in place
        between replays of a captured CUDA graph takes effect at every replay.  The mask is kept, not copied."""
        if _is_torch(warm_start):
            import torch
            if warm_start.dtype not in (torch.bool, torch.uint8) or warm_start.dim() != 1:
                raise ValueError("a warm-start mask must be a 1-D bool or uint8 tensor")
            if warm_start.device.type != "cuda":
                raise ValueError("a torch warm-start mask must be a CUDA tensor (numpy masks go with numpy batches)")
            if warm_start.numel() > 1 and warm_start.stride(0) != 1:
                raise ValueError("a warm-start mask must be contiguous (it is read in place)")
            self.warm_start, self.warm_lanes = True, warm_start
        elif isinstance(warm_start, np.ndarray) and warm_start.ndim > 0:
            if warm_start.dtype not in (np.bool_, np.uint8) or warm_start.ndim != 1:
                raise ValueError("a warm-start mask must be a 1-D bool or uint8 array")
            self.warm_start, self.warm_lanes = True, np.ascontiguousarray(warm_start)
        else:
            self.warm_start, self.warm_lanes = bool(warm_start), None

    def _mask_ptr(self, B: int, dev) -> int:
        """Pointer of the per-lane mask for a batch of B lanes (0: none); refuses a mask that does not fit the call."""
        w = self.warm_lanes
        if w is None:
            return 0
        if w.shape[0] != B:
            raise ValueError(f"warm-start mask has {w.shape[0]} lanes, the batch {B}")
        if dev is None:
            if _is_torch(w):
                raise ValueError("numpy batch with a torch warm-start mask: pass a numpy mask")
            return w.ctypes.data
        if not _is_torch(w) or w.device != dev:
            raise ValueError(f"device batch on {dev} needs a CUDA warm-start mask on the same device")
        return w.data_ptr()

    def contact_vars_start(self) -> int:
        return self.lcs

    # --- state in / out (the reference keeps it private, src/fcc_qp.hpp:147-153)
    def GetState(self):
        return self._state

    def SetState(self, x, mu_x, mu_lambda_c):
        self._state = (x, mu_x, mu_lambda_c)

    def ResetState(self):
        self._state = None

    # ------------------------------------------------------------------
    def Solve(self, Q, b, A_eq, b_eq, friction_coeffs, lb, ub):
        """Batched ``FCCQP::Solve`` (``src/fcc_qp.cpp:114-191``).

        Q ``[B,n,n]``, b ``[B,n]``, A_eq ``[B,m,n]``, b_eq ``[B,m]``; friction_coeffs
        ``[B,nc/3]`` or ``[nc/3]``; lb/ub ``[B,n]`` or ``[n]`` (shared by all QPs).
        Q ``[n,n]`` together with A_eq ``[m,n]`` declares a shared-structure batch (one cost
        matrix and one constraint matrix for all B right-hand sides): the KKT factorizations
        are then cached on the device instead of redone per QP (DESIGN.md section 10).
        """
        if _is_torch(Q):
            self._solve_torch(Q, b, A_eq, b_eq, friction_coeffs, lb, ub)
        else:
            self._solve_numpy(Q, b, A_eq, b_eq, friction_coeffs, lb, ub)

    @staticmethod
    def validate_bounds(lb, ub) -> bool:
        """``lb <= ub`` everywhere (``validate_bounds``, src/constraint_utils.cpp:67-69).  The reference only
        ASSERTS it (src/fcc_qp.cpp:121, compiled out by its own -DNDEBUG release flags); the batched entry points
        do not pay an O(B n) host pass per call for it either -- call this where the check is wanted.  With
        ``lb > ub`` the projection returns ``lb`` (same min/max order as the reference)."""
        if _is_torch(lb):
            return bool((lb <= ub).all().item())
        return bool(np.all(np.asarray(lb) <= np.asarray(ub)))

    def GetSolution(self) -> BatchSolution:
        if self._sol is None:
            raise RuntimeError("GetSolution() before Solve()")
        return self._sol

    # ------------------------------------------------------------------
    def _desc(self, B: int, mem: int) -> nat.BatchDesc:
        d = nat.BatchDesc()
        d.abi_version = nat.ABI_VERSION
        d.batch, d.n, d.m, d.nc, d.lambda_c_start = B, self.n, self.m, self.nc, self.lcs
        d.device, d.memory_space, d.precision = self.device, mem, {"fp64": 0, "fp32_data": 1, "fp32": 2}[self.precision]
        o = self.options
        d.options = nat.Options(int(o.max_iter), int(getattr(o, 'adapt_rho_interval', 0)), float(o.rho), float(o.eps_fcone), float(o.eps_bound), float(o.relaxation))
        st = self.structure
        if st == "dense":
            d.structure = nat.STRUCTURE_DENSE
        elif isinstance(st, (tuple, list)):
            d.structure = nat.STRUCTURE_CAPS
            d.struct_caps[:] = [int(c) for c in st]
        elif st == "auto" and mem == nat.MEM_DEVICE and self._caps is not None:
            d.structure = nat.STRUCTURE_CAPS
            d.struct_caps[:] = list(self._caps)
        elif st in ("auto", "probe"):
            d.structure = nat.STRUCTURE_AUTO
        else:
            raise ValueError("structure must be 'auto', 'probe', 'dense' or a (nr, ndp, nd0) tuple")
        if self.refine:
            d.structure |= nat.STRUCTURE_REFINE
        return d

    def _after_device_call(self, B: int, probed: bool):
        """Bookkeeping of the cached structure bounds ("auto" with device tensors)."""
        if self.structure != "auto":
            return
        info = nat.last_struct_info()
        if probed:
            self._caps = info["caps"] if info["used"] else (self.n, 0, 0)   # (n, 0, 0): nothing to reduce
        self._check_deferred = info["used"]

    def structure_info(self) -> dict:
        """``fccqp_last_struct_info`` of the last launch of this process (synchronise first for ``deferred``)."""
        return nat.last_struct_info()

    def _check_shapes(self, shp, B):
        n, m, nc = self.n, self.m, self.nc
        Q, b, A, beq, mu, lb, ub = shp
        if tuple(Q) == (n, n) and tuple(A) == (m, n):
            Q, A = (B, n, n), (B, m, n)       # shared structure
        if tuple(Q) != (B, n, n) or tuple(b) != (B, n) or tuple(A) != (B, m, n) or tuple(beq) != (B, m):
            raise ValueError(f"expected Q[{B},{n},{n}], b[{B},{n}], A_eq[{B},{m},{n}], b_eq[{B},{m}]; got "
                             f"{tuple(Q)}, {tuple(b)}, {tuple(A)}, {tuple(beq)}")
        # (a longer friction_coeffs vector is accepted like the reference does -- it reads the first nc/3 entries,
        # src/constraint_utils.cpp:27-35 -- the batch stride then skips the rest)
        if not (len(mu) in (1, 2) and mu[-1] >= nc // 3 and (len(mu) == 1 or mu[0] == B)):
            if len(mu) and mu[-1] < nc // 3:
                raise IndexError(f"friction_coeffs has {mu[-1]} entries per QP, need {nc // 3} "
                                 "(reference: std::out_of_range, src/constraint_utils.cpp:32)")
            raise ValueError(f"friction_coeffs must be [{B},{nc // 3}] or [{nc // 3}], got {tuple(mu)}")
        for name, s in (("lb", lb), ("ub", ub)):
            if tuple(s) not in ((B, n), (n,)):
                raise ValueError(f"{name} must be [{B},{n}] or [{n}], got {tuple(s)}")

    def _solve_numpy(self, Q, b, A_eq, b_eq, mu, lb, ub):
        import time
        in_dtype = np.float64 if self.precision == "fp64" else np.float32
        f = lambda a: np.ascontiguousarray(a, dtype=in_dtype)
        Q, b, A_eq, b_eq, mu, lb, ub = map(f, (Q, b, A_eq, b_eq, mu, lb, ub))
        if Q.ndim not in (2, 3):
            raise ValueError("Q must be [B,n,n] (or [n,n] with A_eq [m,n] for a shared-structure batch)")
        shared = Q.ndim == 2
        B = b.shape[0] if shared else Q.shape[0]
        if not shared:
            A_eq = A_eq.reshape(B, self.m, self.n) if A_eq.size == B * self.m * self.n else A_eq
        self._check_shapes([a.shape for a in (Q, b, A_eq, b_eq, mu, lb, ub)], B)
        n, m, nc = self.n, self.m, self.nc
        warm = self.warm_start
        mask = self._mask_ptr(B, None)
        rho = self._rho_ptr(B, None)
        st = self._state
        # Outputs live in solver-owned page-locked buffers (true asynchronous D2H), reused from
        # call to call; x doubles as the carried warm-start state, exactly like the reference's x_.
        ob = self._host_out
        if ob is None or ob["x"].shape != (B, n):
            pe = nat.pinned_empty
            ob = self._host_out = dict(x=pe((B, n), np.float64), mux=pe((B, n), np.float64), muc=pe((B, nc), np.float64),
                                       n_iter=pe((B,), np.int32), status=pe((B,), np.int32), res=pe((4, B), np.float64))
            fresh = True
        else:
            fresh = False
        x, mux, muc = ob["x"], ob["mux"], ob["muc"]
        if warm and st is not None and not _is_torch(st[0]) and st[0].shape == (B, n):
            if st[0] is not x:
                x[...], mux[...], muc[...] = st
        elif warm or fresh:
            # a never-solved reference object warm-starts from the zero state (src/fcc_qp.cpp:48-52)
            x[...] = 0.0; mux[...] = 0.0; muc[...] = 0.0
        n_iter, status, res = ob["n_iter"], ob["status"], ob["res"]
        d = self._desc(B, nat.MEM_HOST)
        d.warm_start = int(warm)
        d.warm_lanes = mask or None
        p = lambda a: a.ctypes.data
        d.Q, d.q_batch_stride, d.q_row_stride, d.q_col_stride = p(Q), (0 if shared else n * n), n, 1
        d.b, d.b_batch_stride = p(b), n
        d.A_eq, d.a_batch_stride, d.a_row_stride, d.a_col_stride = p(A_eq), (0 if shared else m * n), n, 1
        d.b_eq, d.beq_batch_stride = p(b_eq), m
        d.friction_coeffs, d.mu_batch_stride = p(mu), (mu.shape[1] if mu.ndim == 2 else 0)
        d.lb, d.lb_batch_stride = p(lb), (n if lb.ndim == 2 else 0)
        d.ub, d.ub_batch_stride = p(ub), (n if ub.ndim == 2 else 0)
        d.x, d.mu_x, d.mu_lambda_c = p(x), p(mux), p(muc)
        d.n_iter, d.status = p(n_iter), p(status)
        d.res_bounds, d.res_fcone, d.bounds_viol, d.fcone_viol = (p(res[i]) for i in range(4))
        secs = C.c_double(0.0)
        d.device_seconds = C.pointer(secs)
        t0 = time.perf_counter()
        if self.devices is not None:
            devs = (C.c_int32 * len(self.devices))(*self.devices)
            nat.check(nat.lib().fccqp_batch_solve_multi_rho(C.byref(d), rho or None, devs, len(self.devices)))
        else:
            nat.check(nat.lib().fccqp_batch_solve_rho(C.byref(d), rho or None))
        wall = time.perf_counter() - t0
        self._state = (x, mux, muc)
        # zero_copy_outputs: z and the details are views of the solver-owned page-locked buffers,
        # valid until the next Solve(); default: independent copies, like FCCQP::GetSolution.
        cp = (lambda a: a) if self.zero_copy_outputs else (lambda a: a.copy())
        self._sol = BatchSolution(BatchDetails(cp(n_iter), cp(res[0]), cp(res[1]), cp(res[2]), cp(res[3]), cp(status),
                                               wall, secs.value), cp(x))

    def _solve_torch(self, Q, b, A_eq, b_eq, mu, lb, ub):
        import time
        import torch
        dev = Q.device
        if dev.type != "cuda":
            raise ValueError("torch inputs must be CUDA tensors (no CPU solve path); pass numpy arrays for host data")
        self.device = dev.index if dev.index is not None else torch.cuda.current_device()
        in_dtype = torch.float64 if self.precision == "fp64" else torch.float32
        t = lambda a: a if (_is_torch(a) and a.dtype == in_dtype and a.device == dev) else \
            torch.as_tensor(a, dtype=in_dtype, device=dev)
        Q, b, A_eq, b_eq, mu, lb, ub = map(t, (Q, b, A_eq, b_eq, mu, lb, ub))
        if Q.dim() == 2 and A_eq.dim() == 2:      # shared structure: one Q / A_eq, batch stride 0
            Q = Q.unsqueeze(0).expand(b.shape[0], *Q.shape)
            A_eq = A_eq.unsqueeze(0).expand(b.shape[0], *A_eq.shape)
        B = Q.shape[0]
        self._check_shapes([a.shape for a in (Q, b, A_eq, b_eq, mu, lb, ub)], B)
        n, m, nc = self.n, self.m, self.nc
        # vectors must be unit-stride in their last dimension
        cont = lambda a: a if a.stride(-1) == 1 or a.shape[-1] <= 1 else a.contiguous()
        b, b_eq, mu, lb, ub = map(cont, (b, b_eq, mu, lb, ub))
        warm = self.warm_start
        mask = self._mask_ptr(B, dev)
        rho = self._rho_ptr(B, dev)
        st = self._state
        # Outputs and carried state live in solver-owned device tensors, allocated once per (B, device) and reused
        # from call to call (nothing is allocated inside a steady-state Solve).  A cold solve ignores the state
        # on input (the kernel starts from zero duals), so the buffers need no clearing.
        ob = self._dev_out
        if ob is None or ob["x"].shape != (B, n) or ob["x"].device != dev:
            ob = self._dev_out = dict(x=torch.zeros((B, n), dtype=torch.float64, device=dev),
                                      mux=torch.zeros((B, n), dtype=torch.float64, device=dev),
                                      muc=torch.zeros((B, nc), dtype=torch.float64, device=dev),
                                      n_iter=torch.empty(B, dtype=torch.int32, device=dev),
                                      status=torch.empty(B, dtype=torch.int32, device=dev),
                                      res=torch.empty((4, B), dtype=torch.float64, device=dev))
            fresh = True
        else:
            fresh = False
        x, mux, muc = ob["x"], ob["mux"], ob["muc"]
        if warm and st is not None and _is_torch(st[0]) and tuple(st[0].shape) == (B, n) and st[0].device == dev:
            if st[0] is not x:      # state handed in through SetState
                x.copy_(st[0]); mux.copy_(st[1]); muc.copy_(st[2])
        elif warm and not fresh:
            # a never-solved reference object warm-starts from the zero state (src/fcc_qp.cpp:48-52)
            x.zero_(); mux.zero_(); muc.zero_()
        n_iter, status, res = ob["n_iter"], ob["status"], ob["res"]
        if self.structure == "auto" and self._caps is not None and getattr(self, "_check_deferred", False):
            # the previous launch has long been consumed by now: many QPs beyond the cached bounds -> probe again
            if nat.last_struct_info()["deferred"] > B // 16:
                self._caps = None
        d = self._desc(B, nat.MEM_DEVICE)
        probed = (d.structure & ~(nat.STRUCTURE_REFINE | nat.SCHEDULE_LPT)) == nat.STRUCTURE_AUTO
        d.warm_start = int(warm)
        d.warm_lanes = mask or None
        if self.schedule_from_previous and not fresh:
            d.structure |= nat.SCHEDULE_LPT
        bs = lambda a, full_ndim: int(a.stride(0)) if a.dim() == full_ndim and B > 1 else (
            int(a.stride(0)) if a.dim() == full_ndim else 0)
        d.Q, d.q_batch_stride, d.q_row_stride, d.q_col_stride = Q.data_ptr(), bs(Q, 3), int(Q.stride(1)), int(Q.stride(2))
        d.b, d.b_batch_stride = b.data_ptr(), bs(b, 2)
        d.A_eq, d.a_batch_stride = A_eq.data_ptr(), bs(A_eq, 3)
        d.a_row_stride, d.a_col_stride = (int(A_eq.stride(1)), int(A_eq.stride(2))) if m > 0 else (n, 1)
        d.b_eq, d.beq_batch_stride = b_eq.data_ptr(), bs(b_eq, 2)
        d.friction_coeffs, d.mu_batch_stride = mu.data_ptr(), bs(mu, 2)
        d.lb, d.lb_batch_stride = lb.data_ptr(), bs(lb, 2)
        d.ub, d.ub_batch_stride = ub.data_ptr(), bs(ub, 2)
        d.x, d.mu_x, d.mu_lambda_c = x.data_ptr(), mux.data_ptr(), muc.data_ptr()
        d.n_iter, d.status = n_iter.data_ptr(), status.data_ptr()
        d.res_bounds, d.res_fcone, d.bounds_viol, d.fcone_viol = (res[i].data_ptr() for i in range(4))
        d.stream = torch.cuda.current_stream(dev).cuda_stream
        secs = C.c_double(0.0)
        if self.time_kernel:
            d.device_seconds = C.pointer(secs)
        t0 = time.perf_counter()
        with torch.cuda.device(dev):
            nat.check(nat.lib().fccqp_batch_solve_rho(C.byref(d), rho or None))
        wall = time.perf_counter() - t0
        self._after_device_call(B, probed)
        # keep the inputs alive until the (possibly asynchronous) launch has consumed them
        self._keepalive = (Q, b, A_eq, b_eq, mu, lb, ub)
        self._mask_keepalive = (self.warm_lanes, self.rho_lanes)
        self._state = (x, mux, muc)
        # zero_copy_outputs: z and the details are the solver-owned tensors themselves, valid until the next Solve();
        # default: independent copies, like FCCQP::GetSolution
        cp = (lambda a: a) if self.zero_copy_outputs else (lambda a: a.clone())
        self._sol = BatchSolution(BatchDetails(cp(n_iter), cp(res[0]), cp(res[1]), cp(res[2]), cp(res[3]), cp(status),
                                               wall, secs.value), cp(x))


    # ------------------------------------------------------------------
    def Polish(self):
        """Opt-in solution polish of the batch just solved (extension: NOT in the reference; include/fccqp.h,
        fccqp_polish_prepare / _finish).  Device path only: call after ``Solve`` on torch CUDA tensors in FP64.  The active
        set is guessed from the solver's state, the resulting equality-constrained QPs (same n, m) are solved by a second
        batched launch (nc = 0, no bounds: the KKT solve), and a QP takes the polished point only if that solve succeeded
        and the point satisfies every bound and friction cone to the solver's tolerances and is not worse in objective
        than the ADMM iterate by more than ``polish_objective_slack`` (1e-3, relative).  Updates ``GetSolution()``:
        ``z``, ``bounds_viol``, ``friction_cone_viol`` of the accepted QPs, ``details.polished`` [B] = 1 / 0; iteration
        counts, residuals, status and the carried duals are left as the ADMM solve wrote them."""
        import torch
        if self._dev_out is None or getattr(self, "_keepalive", None) is None or self._sol is None or not _is_torch(self._sol.z):
            raise RuntimeError("Polish() needs a preceding Solve() on torch CUDA tensors (device path)")
        if self.precision != "fp64":
            raise ValueError("Polish() is an FP64 path")
        Q, b, A_eq, b_eq, mu, lb, ub = self._keepalive
        ob = self._dev_out
        n, m, nc = self.n, self.m, self.nc
        B = ob["x"].shape[0]
        dev = ob["x"].device
        # dense row-major per QP (batch stride 0 = shared is fine)
        dense = lambda a: a if (a.stride(-1) == 1 and a.stride(-2) == a.shape[-1]) or a.numel() == 0 else a.contiguous()
        Q, A_eq = dense(Q), dense(A_eq)
        pb = getattr(self, "_polish_buf", None)
        if pb is None or pb["Qp"].shape[0] != B or pb["Qp"].device != dev:
            f = lambda *s_: torch.empty(s_, dtype=torch.float64, device=dev)
            pb = self._polish_buf = dict(Qp=f(B, n, n), bp=f(B, n), Ap=f(B, m, n), beqp=f(B, m), rot=f(B, max(nc // 3, 1), 4),
                                         flag=torch.empty(B, dtype=torch.int32, device=dev),
                                         inf_lo=torch.full((n,), -float("inf"), dtype=torch.float64, device=dev),
                                         inf_hi=torch.full((n,), float("inf"), dtype=torch.float64, device=dev),
                                         no_mu=torch.empty((0,), dtype=torch.float64, device=dev))
            inner = FCCQPBatch(n, m, 0, 0, device=self.device)
            inner.zero_copy_outputs = True
            inner.time_kernel = False
            inner.refine = True       # the polish is about accuracy: one refinement step of the reduced pre-solve (7e-11 instead of 1.2e-7)
            pb["inner"] = inner
        inner = pb["inner"]
        inner.set_options(self.options)
        inner.structure = self.structure if isinstance(self.structure, str) else "auto"
        d = nat.PolishDesc()
        d.abi_version = nat.ABI_VERSION
        d.batch, d.n, d.m, d.nc, d.lambda_c_start, d.device = B, n, m, nc, self.lcs, self.device
        d.eps_fcone, d.eps_bound = float(self.options.eps_fcone), float(self.options.eps_bound)
        d.eps_objective = float(getattr(self, "polish_objective_slack", 1e-3))
        bs = lambda a, full_ndim: int(a.stride(0)) if a.dim() == full_ndim else 0
        d.Q, d.q_batch_stride = Q.data_ptr(), bs(Q, 3)
        d.b, d.b_batch_stride = b.data_ptr(), bs(b, 2)
        d.A_eq, d.a_batch_stride = A_eq.data_ptr(), bs(A_eq, 3)
        d.b_eq, d.beq_batch_stride = b_eq.data_ptr(), bs(b_eq, 2)
        d.friction_coeffs, d.mu_batch_stride = mu.data_ptr(), bs(mu, 2)
        d.lb, d.lb_batch_stride = lb.data_ptr(), bs(lb, 2)
        d.ub, d.ub_batch_stride = ub.data_ptr(), bs(ub, 2)
        d.x, d.mu_x, d.mu_lambda_c = ob["x"].data_ptr(), ob["mux"].data_ptr(), ob["muc"].data_ptr()
        d.Qp, d.bp, d.Ap, d.beqp, d.rot = (pb[k].data_ptr() for k in ("Qp", "bp", "Ap", "beqp", "rot"))
        d.stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            nat.check(nat.lib().fccqp_polish_prepare(C.byref(d)))
            inner.set_warm_start(False)
            inner.Solve(pb["Qp"], pb["bp"], pb["Ap"], pb["beqp"], pb["no_mu"], pb["inf_lo"], pb["inf_hi"])
            y = inner.GetSolution()
            d.y, d.y_status = y.z.data_ptr(), y.details.solve_status.data_ptr()
            res = ob["res"]
            d.z, d.bounds_viol, d.fcone_viol = ob["x"].data_ptr(), res[2].data_ptr(), res[3].data_ptr()
            d.polished = pb["flag"].data_ptr()
            nat.check(nat.lib().fccqp_polish_finish(C.byref(d)))
        cp = (lambda a: a) if self.zero_copy_outputs else (lambda a: a.clone())
        det = self._sol.details
        self._sol = BatchSolution(dataclasses.replace(det, bounds_viol=cp(res[2]), friction_cone_viol=cp(res[3]),
                                                      polished=cp(pb["flag"])), cp(ob["x"]))
        return self._sol


class FCCQPBatchCpp:
    """The same batched surface as a thin shim over the C++ class ``fcc_qp::FCCQPBatch`` (``include/fcc_qp.hpp``) as
    bound in the pybind11 module (``fcc_qp_solver.FCCQPBatch``): numpy stacks go to its host path, anything with
    ``__dlpack__`` (torch CUDA tensors, cupy arrays) to its device path -- zero-copy, asynchronous on ``stream``,
    outputs and carried state in tensors allocated once and reused.  No option of ``FCCQPBatch`` beyond the
    reference's own is mirrored here (precision modes, structure caps, pinned zero-copy outputs stay there)."""

    def __init__(self, num_vars: int, num_equality_constraints: int, nc: int, lambda_c_start: int, device=0):
        from . import fcc_qp_solver as mod
        self._mod = mod
        self.n, self.m, self.nc, self.lcs = int(num_vars), int(num_equality_constraints), int(nc), int(lambda_c_start)
        self._s = mod.FCCQPBatch(self.n, self.m, self.nc, self.lcs, list(device)) if isinstance(device, (list, tuple)) \
            else mod.FCCQPBatch(self.n, self.m, self.nc, self.lcs, int(device))
        self._out = None
        self._sol = None
        self._mask = None      # torch per-lane mask of the device path (SolveDLPack's warm_lanes)
        self._rho = None       # torch per-lane rho of the device path (SolveDLPack's rho)
        self.time_kernel = False

    def set_rho(self, rho):
        """A float, or a per-lane [B] rho: numpy / sequence for host stacks (the C++ object keeps a copy and writes the
        final rho into it: ``rho_lanes``), a contiguous CUDA float64 tensor for device ones (read and written in place)."""
        self._rho = None
        if _is_torch(rho):
            self._rho = rho
        elif isinstance(rho, (list, tuple)) or (isinstance(rho, np.ndarray) and rho.ndim > 0):
            self._s.set_rho(np.asarray(rho, dtype=np.float64))
        else:
            self._s.set_rho(float(rho))

    @property
    def rho_lanes(self):
        return self._rho if self._rho is not None else self._s.rho_lanes
    def set_max_iter(self, n): self._s.set_max_iter(int(n))

    def set_warm_start(self, warm_start):
        """A bool, or a per-lane [B] mask: numpy / sequence for host stacks, a CUDA bool / uint8 tensor for device ones."""
        self._mask = None
        if _is_torch(warm_start):
            self._mask = warm_start
            self._s.set_warm_start(True)
        elif isinstance(warm_start, (list, tuple)) or (isinstance(warm_start, np.ndarray) and warm_start.ndim > 0):
            self._s.set_warm_start(np.asarray(warm_start, dtype=np.uint8))
        else:
            self._s.set_warm_start(bool(warm_start))
    def contact_vars_start(self): return self.lcs

    def set_options(self, opt):
        o = self._mod.FCCQPOptions()
        for k in ("max_iter", "rho", "eps_fcone", "eps_bound", "relaxation", "adapt_rho_interval"):
            if hasattr(opt, k):
                setattr(o, k, getattr(opt, k))
        self._s.set_options(o)

    def Solve(self, Q, b, A_eq, b_eq, friction_coeffs, lb, ub):
        if not hasattr(Q, "__dlpack__") or isinstance(Q, np.ndarray):
            self._s.Solve(Q, b, A_eq, b_eq, friction_coeffs, lb, ub)
            r = self._s.GetSolution()
            self._sol = BatchSolution(BatchDetails(r.n_iter, r.eps_bounds, r.eps_friction_cone, r.bounds_viol,
                                                   r.friction_cone_viol, r.solve_status, r.solve_time, r.solve_time), r.z)
            return
        import torch
        B, dev = int(b.shape[0]), b.device
        o = self._out
        if o is None or o[0].shape[0] != B or o[0].device != dev:
            f64 = dict(dtype=torch.float64, device=dev)
            o = self._out = (torch.zeros((B, self.n), **f64), torch.zeros((B, self.n), **f64), torch.zeros((B, self.nc), **f64),
                             torch.empty(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev),
                             torch.empty((4, B), **f64))
        mu = friction_coeffs if hasattr(friction_coeffs, "__dlpack__") and not isinstance(friction_coeffs, np.ndarray) \
            else torch.as_tensor(np.asarray(friction_coeffs, dtype=np.float64), device=dev)
        with torch.cuda.device(dev):
            secs = self._s.SolveDLPack(Q, b, A_eq, b_eq, mu, lb, ub, *o,
                                       stream=torch.cuda.current_stream(dev).cuda_stream, time_kernel=self.time_kernel,
                                       warm_lanes=self._mask, rho=self._rho)
        self._keepalive = (Q, b, A_eq, b_eq, mu, lb, ub, self._mask, self._rho)
        x, _, _, n_iter, status, det = o
        self._sol = BatchSolution(BatchDetails(n_iter, det[0], det[1], det[2], det[3], status, secs, secs), x)

    def GetSolution(self) -> BatchSolution:
        if self._sol is None:
            raise RuntimeError("GetSolution() before Solve()")
        return self._sol


def solve_batch(Q, b, A_eq, b_eq, friction_coeffs, lb, ub, nc: int, lambda_c_start: int,
                options=None, device: int = 0) -> BatchSolution:
    """One-shot cold batched solve; dimensions are taken from the array shapes."""
    B, n, _ = Q.shape
    m = A_eq.shape[1]
    s = FCCQPBatch(n, m, nc, lambda_c_start, device=device)
    if options is not None:
        s.set_options(options)
    s.Solve(Q, b, A_eq, b_eq, friction_coeffs, lb, ub)
    return s.GetSolution()
