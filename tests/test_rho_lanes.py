"""Per-lane rho without a GPU (fccqp_batch_solve_rho, FCCQPBatch.set_rho(array)): the C entry points link and refuse a bad
host array before touching a device, the Python and C++ front ends refuse arrays that do not fit the call, and the C
restatement reports the rho a solve ended with -- carrying it into the next warm solve changes nothing but the starting
rho."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rho_oracle
from conftest import LOG_OPTS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def nat():
    from fcc_qp_b200 import _native
    return _native


def test_c_caller_links_both_entry_points_and_bad_host_rho_is_refused(nat, tmp_path):
    """A C caller of the header: both new symbols resolve at link time, and a host array with an entry that is zero,
    negative or NaN is refused with FCCQP_E_INVALID before any device is needed."""
    src = tmp_path / "rho.c"
    src.write_text(r'''
#include <math.h>
#include <stdio.h>
#include <string.h>
#include "fccqp.h"
int main(void) {
  enum { B = 3, n = 4, m = 1 };
  static double Q[B * n * n], b[B * n], A[B * m * n], beq[B * m], lb[B * n], ub[B * n], x[B * n], mux[B * n];
  fccqp_batch_desc d;
  memset(&d, 0, sizeof d);
  d.abi_version = FCCQP_ABI_VERSION; d.batch = B; d.n = n; d.m = m;
  fccqp_default_options(&d.options);
  d.memory_space = FCCQP_MEM_HOST;
  d.Q = Q; d.q_batch_stride = n * n; d.q_row_stride = n; d.q_col_stride = 1;
  d.b = b; d.b_batch_stride = n; d.A_eq = A; d.a_batch_stride = m * n; d.a_row_stride = n; d.a_col_stride = 1;
  d.b_eq = beq; d.beq_batch_stride = m; d.lb = lb; d.lb_batch_stride = n; d.ub = ub; d.ub_batch_stride = n;
  d.x = x; d.mu_x = mux;
  const double bad[3] = {0.0, -1.0, NAN};
  int32_t dev = 0;
  for (int k = 0; k < 3; ++k) {
    double rho[B] = {1e-3, 1e-3, 1e-3};
    rho[1] = bad[k];
    const int r1 = fccqp_batch_solve_rho(&d, rho);
    const int r2 = fccqp_batch_solve_multi_rho(&d, rho, &dev, 1);
    printf("%d %d %d\n", r1, r2, strstr(fccqp_last_error(), "rho[1]") != NULL);
  }
  return 0;
}
''')
    exe = tmp_path / "rho"
    libdir = os.path.join(ROOT, "fcc_qp_b200")
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir, "-lfccqp_b200",
                           f"-Wl,-rpath,{libdir}", "-lm", "-o", str(exe)])
    lines = subprocess.check_output([str(exe)], text=True).split("\n")
    for line in lines[:3]:
        assert [int(v) for v in line.split()] == [nat.E_INVALID, nat.E_INVALID, 1], lines


def test_ctypes_bindings_resolve(nat):
    lib = nat.lib()
    for name in ("fccqp_batch_solve_rho", "fccqp_batch_solve_multi_rho"):
        assert name in nat.EXPORTS
        assert getattr(lib, name).argtypes is not None


def test_python_set_rho_checks():
    import torch
    from fcc_qp_b200.batch import FCCQPBatch
    s = FCCQPBatch(6, 0, 6, 0)
    for bad in (np.ones(4, np.float32), np.ones((2, 2)), np.ones(8)[::2], np.array([1e-3, 0.0]), np.array([1e-3, -1.0]),
                np.array([1e-3, np.nan]), np.array([1e-3, np.inf]), torch.ones(4, dtype=torch.float32),
                torch.ones((2, 2), dtype=torch.float64), torch.ones(4, dtype=torch.float64)):   # (the last: not CUDA)
        with pytest.raises(ValueError):
            s.set_rho(bad)
    with pytest.raises(ValueError):
        s.set_rho(0.0)
    r = np.full(3, 1e-3)
    s.set_rho(r)
    assert s.rho_lanes is r                     # kept, not copied: every Solve reads and writes it in place
    z = lambda *shape: np.zeros(shape)
    with pytest.raises(ValueError, match="3 lanes, the batch 2"):     # wrong length: refused before any launch
        s.Solve(z(2, 6, 6), z(2, 6), z(2, 0, 6), z(2, 0), z(2, 2), z(6), z(6))
    r2 = np.full(2, 1e-3)
    s.set_rho(r2)
    r2[1] = -1.0                                # changed in place after set_rho: refused at Solve
    with pytest.raises(ValueError, match="finite and > 0"):
        s.Solve(z(2, 6, 6), z(2, 6), z(2, 0, 6), z(2, 0), z(2, 2), z(6), z(6))
    r2[1] = 1e-3
    assert s._rho_ptr(2, None) == r2.ctypes.data
    with pytest.raises(ValueError, match="CUDA per-lane rho"):        # numpy array with a device batch
        s._rho_ptr(2, torch.device("cuda", 0))
    s.rho_lanes = torch.ones(2, dtype=torch.float64)                  # (a torch array with a numpy batch)
    with pytest.raises(ValueError, match="numpy batch with a torch"):
        s._rho_ptr(2, None)
    s.set_rho(r2)
    s.set_rho(2e-3)                             # a float: one rho for every lane, the array is dropped
    assert s.rho_lanes is None and s.options.rho == 2e-3


def test_pybind_set_rho_checks():
    from fcc_qp_b200 import fcc_qp_solver as mod
    s = mod.FCCQPBatch(6, 0, 6, 0)
    s.set_rho(1e-3)
    assert s.rho_lanes.size == 0
    s.set_rho([1e-3, 2e-3, 3e-3])
    assert np.array_equal(s.rho_lanes, [1e-3, 2e-3, 3e-3])
    with pytest.raises(ValueError, match="rho_lanes has 3 entries"):   # std::invalid_argument before the C call
        s.Solve(np.zeros((2, 6, 6)), np.zeros((2, 6)), np.zeros((2, 0, 6)), np.zeros((2, 0)), np.zeros((2, 2)),
                np.zeros(6), np.zeros(6))
    for bad in ([1e-3, 0.0], [np.nan], np.zeros((2, 2))):
        with pytest.raises(ValueError):
            s.set_rho(bad)
    s.set_rho(1e-3)
    assert s.rho_lanes.size == 0


def test_cpp_header_compiles_with_the_rho_api(tmp_path):
    src = tmp_path / "r.cpp"
    src.write_text(r'''
#include "fcc_qp.hpp"
int main() {
  fcc_qp::FCCQPBatch b(6, 0, 6, 0);
  b.set_rho(std::vector<double>{1e-3, 2e-3});
  const std::vector<double>& r = b.rho_lanes();
  (void)r;
  b.set_rho(1e-3);
  void (fcc_qp::FCCQPBatch::*dev)(int, const fcc_qp::FCCQPBatchDeviceIO&, double*, const uint8_t*, double*) =
      &fcc_qp::FCCQPBatch::SolveDevice;
  (void)dev;
  return 0;
}
''')
    subprocess.check_call(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])


# ---- the restatement's record of the final rho (tests/rho_oracle.py)
@pytest.fixture()
def port(tmp_path_factory):
    o = rho_oracle.load(tmp_path_factory.mktemp("rho_oracle"))
    yield o
    o.set_adaptive_rho(0)


def set_rho(s, rho):
    """FCCQP::set_rho on a restatement object: the options of LOG_OPTS with another rho."""
    s.set_options(LOG_OPTS["max_iter"], rho, LOG_OPTS["eps_fcone"], LOG_OPTS["eps_bound"])


def _solve(s, q):
    s.Solve(q["Q"], q["b"], q["A_eq"], q["b_eq"], q["friction_coeffs"], q["lb"], q["ub"])
    return s.GetSolution()


def test_oracle_last_rho(port, walking_log):
    idx = range(0, 2019, 40)
    s = port.solver(walking_log.n, walking_log.m, walking_log.nc, walking_log.lambda_c_start)
    s.set_options(**LOG_OPTS)
    for i in idx:                                   # adaptive rho off: the rho the solve was given
        _solve(s, walking_log.qp(i))
        assert port.last_rho() == LOG_OPTS["rho"]
    set_rho(s, 3e-4)
    _solve(s, walking_log.qp(0))
    assert port.last_rho() == 3e-4
    port.set_adaptive_rho(5)
    set_rho(s, LOG_OPTS["rho"])
    moved = []
    for i in idx:
        r = _solve(s, walking_log.qp(i))
        moved.append(port.last_rho() != LOG_OPTS["rho"])
        if r["n_iter"] < 5:                         # no rebalance before iteration 5
            assert not moved[-1]
    assert any(moved)


def test_oracle_carried_rho_changes_only_the_starting_rho(port, walking_log):
    """Warm-sequential over the log with adaptive rho every 5 iterations, twice: restarting each solve at options.rho, and
    carrying the rho the previous solve ended with (set_rho(last_rho)).  Up to and including the first solve whose rho
    moved the two runs are bit-identical -- they start every solve from the same rho -- and after it they part ways."""
    port.set_adaptive_rho(5)
    n, m, nc, lcs = walking_log.n, walking_log.m, walking_log.nc, walking_log.lambda_c_start
    runs = {}
    for carry in (False, True):
        s = port.solver(n, m, nc, lcs)
        s.set_options(**LOG_OPTS)
        s.set_warm_start(True)
        out = []
        for i in range(400):
            r = _solve(s, walking_log.qp(i))
            out.append((r["z"].tobytes(), r["n_iter"], port.last_rho(), s.get_state()[1].tobytes()))
            if carry:
                set_rho(s, port.last_rho())
        runs[carry] = out
    first = next(i for i, o in enumerate(runs[False]) if o[2] != LOG_OPTS["rho"])
    assert runs[True][: first + 1] == runs[False][: first + 1]
    assert runs[True][first + 1:] != runs[False][first + 1:]
    later = [i for i in range(first + 1, 400) if runs[True][i] != runs[False][i]]
    print(f"first moved rho at solve {first}; {len(later)} of {399 - first} later solves differ")


def test_recording_build_computes_what_the_restatement_computes(port, walking_log):
    """The library of tests/rho_oracle.py adds statements that record rho and nothing else: over a batch that adapts,
    its outputs are those of the checked-in restatement, bit for bit."""
    import oracle
    qp = walking_log.take(np.arange(0, 2019, 4))
    plain = oracle.Oracle("port")
    try:
        for o in (port, plain):
            o.set_adaptive_rho(5)
        a = port.solve_batch(qp, warm_mode=1, nthreads=1, **LOG_OPTS)
        b = plain.solve_batch(qp, warm_mode=1, nthreads=1, **LOG_OPTS)
    finally:
        plain.set_adaptive_rho(0)
    for k in ("z", "n_iter", "status", "res_bounds", "res_fcone", "bounds_viol", "fcone_viol"):
        assert a[k].tobytes() == b[k].tobytes(), k
    assert (a["n_iter"] >= 5).any()
