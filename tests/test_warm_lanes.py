"""Per-lane cold or warm start without a GPU: the C ABI refuses a mask without the state it needs before touching a
device, the descriptor's new field sits where the header puts it, and the Python and C++ front ends refuse a mask that
does not fit the call before any launch."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def nat():
    from fcc_qp_b200 import _native
    return _native


def _desc(nat, keep, B=4, n=6, m=2, nc=3):
    d = nat.BatchDesc()
    d.abi_version = nat.ABI_VERSION
    d.batch, d.n, d.m, d.nc, d.lambda_c_start = B, n, m, nc, 0
    d.options = nat.Options(100, 0, 1e-3, 1e-3, 1e-6, 1.0)
    arr = lambda *shape: keep.append(np.zeros(shape)) or keep[-1].ctypes.data
    d.Q, d.q_batch_stride, d.q_row_stride, d.q_col_stride = arr(B, n, n), n * n, n, 1
    d.b, d.b_batch_stride = arr(B, n), n
    d.A_eq, d.a_batch_stride, d.a_row_stride, d.a_col_stride = arr(B, m, n), m * n, n, 1
    d.b_eq, d.beq_batch_stride = arr(B, m), m
    d.friction_coeffs, d.mu_batch_stride = arr(B, 1), 1
    d.lb, d.lb_batch_stride = arr(B, n), n
    d.ub, d.ub_batch_stride = arr(B, n), n
    d.x, d.mu_x, d.mu_lambda_c = arr(B, n), arr(B, n), arr(B, nc)
    mask = np.array([1, 0, 1, 0], np.uint8)
    keep.append(mask)
    d.warm_lanes = mask.ctypes.data
    return d


@pytest.mark.parametrize("missing", ["mu_x", "mu_lambda_c"])
@pytest.mark.parametrize("memory_space", [0, 1])
def test_mask_needs_the_carried_duals(nat, missing, memory_space):
    keep = []
    d = _desc(nat, keep)
    d.memory_space = memory_space
    setattr(d, missing, None)
    lib = nat.lib()
    assert lib.fccqp_batch_solve(C.byref(d)) == nat.E_INVALID
    assert b"warm_lanes" in lib.fccqp_last_error()
    devs = (C.c_int32 * 1)(0)
    if memory_space == 0:
        assert lib.fccqp_batch_solve_multi(C.byref(d), devs, 1) == nat.E_INVALID
        assert b"warm_lanes" in lib.fccqp_last_error()


def test_descriptor_field_matches_the_header(nat, tmp_path):
    src = tmp_path / "abi.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "fccqp.h"
int main(void) {
  printf("%zu %zu %zu\n", offsetof(fccqp_batch_desc, warm_lanes), sizeof(((fccqp_batch_desc*)0)->warm_lanes), sizeof(fccqp_batch_desc));
  return 0;
}
''')
    exe = tmp_path / "abi"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    off, size, total = (int(v) for v in subprocess.check_output([str(exe)], text=True).split())
    assert (off, size, total) == (nat.BatchDesc.warm_lanes.offset, C.sizeof(C.c_void_p), C.sizeof(nat.BatchDesc))
    assert nat.BatchDesc.warm_lanes.offset > nat.BatchDesc.struct_caps.offset     # appended: earlier fields stay put
    assert nat.ABI_VERSION == 5


def test_python_mask_checks():
    import torch
    from fcc_qp_b200.batch import FCCQPBatch
    s = FCCQPBatch(6, 0, 6, 0)
    for bad in (np.zeros(4, np.float64), np.zeros((2, 2), bool), np.zeros(4, np.int32), torch.zeros(4, dtype=torch.bool),
                torch.zeros(4, dtype=torch.float32)):
        with pytest.raises(ValueError):
            s.set_warm_start(bad)
    s.set_warm_start(np.array([True, False, True]))
    assert s.warm_start and s.warm_lanes is not None
    z = lambda *shape: np.zeros(shape)
    # wrong length: refused before any launch (and before any device is touched)
    with pytest.raises(ValueError, match="3 lanes, the batch 2"):
        s.Solve(z(2, 6, 6), z(2, 6), z(2, 0, 6), z(2, 0), z(2, 2), z(6), z(6))
    s.set_warm_start(np.zeros(2, np.uint8))
    assert s._mask_ptr(2, None) == s.warm_lanes.ctypes.data
    s.set_warm_start(True)
    assert s.warm_start is True and s.warm_lanes is None
    s.set_warm_start(np.bool_(False))      # a numpy scalar is a plain flag
    assert s.warm_start is False and s.warm_lanes is None


def test_pybind_mask_checks():
    from fcc_qp_b200 import fcc_qp_solver as mod
    s = mod.FCCQPBatch(6, 0, 6, 0)
    s.set_warm_start(True)
    s.set_warm_start([1, 0, 1])
    s.set_warm_start(np.array([True, False, True]))
    with pytest.raises(ValueError, match="warm_lanes has 3 entries"):   # std::invalid_argument before the C call
        s.Solve(np.zeros((2, 6, 6)), np.zeros((2, 6)), np.zeros((2, 0, 6)), np.zeros((2, 0)), np.zeros((2, 2)),
                np.zeros(6), np.zeros(6))
    with pytest.raises(ValueError):
        s.set_warm_start(np.zeros((2, 2)))


def test_cpp_header_compiles_with_the_mask_api(tmp_path):
    src = tmp_path / "m.cpp"
    src.write_text(r'''
#include "fcc_qp.hpp"
int main() {
  fcc_qp::FCCQPBatch b(6, 0, 6, 0);
  b.set_warm_start(std::vector<uint8_t>{1, 0, 1});
  b.set_warm_start(false);
  fcc_qp::FCCQPBatchDeviceIO io;
  (void)io;
  void (fcc_qp::FCCQPBatch::*dev)(int, const fcc_qp::FCCQPBatchDeviceIO&, double*, const uint8_t*) = &fcc_qp::FCCQPBatch::SolveDevice;
  (void)dev;
  return 0;
}
''')
    subprocess.check_call(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])
