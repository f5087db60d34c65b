"""Host-side logic and the drop-in boundary, without a GPU: the C ABI library loads and exports
every symbol include/fccqp.h declares, argument validation mirrors the reference's error
behaviour, and there is no CPU fallback (compute calls fail loudly without a device)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def nat():
    from fcc_qp_b200 import build
    build.build_all()
    from fcc_qp_b200 import _native
    return _native


def test_header_symbols_exported(nat):
    hdr = open(os.path.join(ROOT, "include", "fccqp.h")).read()
    declared = set(re.findall(r"\b(fccqp_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(nat.EXPORTS), declared ^ set(nat.EXPORTS)
    lib = nat.lib()
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.fccqp_abi_version() == nat.ABI_VERSION


def test_struct_layout_matches_header(nat):
    # fccqp_options: 2 x int32 + 4 x double (ABI 2: + relaxation); fccqp_details: 2 x int32 + 6 x double
    assert C.sizeof(nat.Options) == 40 and C.sizeof(nat.Details) == 56
    o = nat.Options()
    nat.lib().fccqp_default_options(C.byref(o))
    assert (o.max_iter, o.rho, o.eps_fcone, o.eps_bound) == (1000, 1e-6, 1e-3, 1e-6)  # src/fcc_qp.hpp:30-35
    assert o.relaxation == 1.0                                                        # extension: 1 = the reference


def _has_gpu(nat):
    return nat.lib().fccqp_device_count() > 0


def test_no_cpu_fallback(nat):
    """Without a CUDA device construction fails with FCCQP_E_CUDA -- nothing is solved on the CPU."""
    if _has_gpu(nat):
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    rc = nat.lib().fccqp_create(60, 38, 12, 38, 0, C.byref(h))
    assert rc == nat.E_CUDA and b"no CPU fallback" in nat.lib().fccqp_last_error()
    from fcc_qp_b200.batch import FCCQPBatch
    s = FCCQPBatch(3, 0, 3, 0)
    with pytest.raises(nat.FCCQPError) as e:
        s.Solve(np.eye(3)[None], np.zeros((1, 3)), np.zeros((1, 0, 3)), np.zeros((1, 0)), [0.5],
                np.full(3, -np.inf), np.full(3, np.inf))
    assert e.value.code == nat.E_CUDA
    import fcc_qp_b200
    with pytest.raises(RuntimeError):
        fcc_qp_b200.FCCQP(60, 38, 12, 38)


def test_dimension_validation(nat):
    h = C.c_void_p()
    lib = nat.lib()
    assert lib.fccqp_create(10, 2, 4, 0, 0, C.byref(h)) == nat.E_INVALID   # nc % 3 != 0 (fcc_qp.cpp:32)
    assert lib.fccqp_create(10, 2, 6, 6, 0, C.byref(h)) == nat.E_INVALID   # lambda_c_start + nc > n (fcc_qp.cpp:33)
    d = nat.BatchDesc()
    d.abi_version = nat.ABI_VERSION
    d.batch, d.n, d.m, d.nc, d.lambda_c_start = 4, 10, 2, 6, 6
    d.options = nat.Options(100, 0, 1e-3, 1e-3, 1e-6)
    assert lib.fccqp_batch_solve(C.byref(d)) == nat.E_INVALID
    d.lambda_c_start = 0
    d.options = nat.Options(100, 0, -1.0, 1e-3, 1e-6)                       # rho <= 0 (fcc_qp.hpp:76)
    assert lib.fccqp_batch_solve(C.byref(d)) == nat.E_INVALID
    d.options = nat.Options(100, 0, 1e-3, 1e-3, 1e-6)
    assert lib.fccqp_batch_solve(C.byref(d)) == nat.E_INVALID               # null pointers
    d.abi_version = 99
    assert lib.fccqp_batch_solve(C.byref(d)) == nat.E_INVALID


def test_python_surface_matches_reference_binding():
    """Names bound in src/main.cpp:22-54."""
    import fcc_qp_b200 as f
    o = f.FCCQPOptions()
    assert (o.max_iter, o.rho, o.eps_fcone, o.eps_bound) == (1000, 1e-6, 1e-3, 1e-6)
    for a in ("n_iter", "eps_bounds", "eps_friction_cone", "bounds_viol", "friction_cone_viol", "solve_time",
              "factorization_time"):
        assert hasattr(f.FCCQPDetails, a)
    for a in ("details", "z"):
        assert hasattr(f.FCCQPSolution, a)
    for a in ("set_rho", "set_max_iter", "set_warm_start", "set_options", "Solve", "GetSolution"):
        assert hasattr(f.FCCQP, a)
    import fcc_qp  # drop-in alias of the reference package name
    assert fcc_qp.FCCQP is f.FCCQP and fcc_qp.FCCQPOptions is f.FCCQPOptions


def test_batch_argument_checks():
    from fcc_qp_b200.batch import FCCQPBatch
    with pytest.raises(ValueError):
        FCCQPBatch(10, 2, 4, 0)
    with pytest.raises(ValueError):
        FCCQPBatch(10, 2, 6, 6)
    s = FCCQPBatch(6, 0, 6, 0)
    z = lambda *s_: np.zeros(s_)
    with pytest.raises(IndexError):   # too few friction coefficients (std::out_of_range in the reference)
        s.Solve(z(2, 6, 6), z(2, 6), z(2, 0, 6), z(2, 0), z(2, 1), z(6), z(6))
    with pytest.raises(ValueError):
        s.Solve(z(2, 6, 5), z(2, 6), z(2, 0, 6), z(2, 0), z(2, 2), z(6), z(6))
    with pytest.raises(ValueError):
        s.set_rho(0.0)
    with pytest.raises(ValueError):
        s.set_max_iter(0)
    with pytest.raises(ValueError):
        FCCQPBatch(6, 0, 6, 0, precision="fp16")
    for prec, code in (("fp64", 0), ("fp32_data", 1), ("fp32", 2)):     # fccqp_precision of include/fccqp.h
        assert FCCQPBatch(6, 0, 6, 0, precision=prec)._desc(1, 0).precision == code


def test_compact_log_roundtrip(tmp_path, walking_log):
    from fcc_qp_b200.logdata import load_compact, save_compact
    sub = walking_log.take(np.arange(0, 2019, 101))
    p = str(tmp_path / "sub.npz")
    save_compact(sub, p)
    back = load_compact(p)
    for k in ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub"):
        assert np.array_equal(getattr(sub, k), getattr(back, k))
    assert (walking_log.n, walking_log.m, walking_log.nc, walking_log.lambda_c_start, walking_log.batch) == (60, 38, 12, 38, 2019)
    t = walking_log.tile(5000)
    assert t.batch == 5000 and np.array_equal(t.Q[2019], walking_log.Q[0])


def test_compact_log_is_bit_exact_copy_of_reference_log(walking_log):
    """The stacked arrays of the reference's pickled log (99 MB, not shipped) hash to the digests that
    tests/golden/make_walking_log.py stored from it; the compact copy must hash the same."""
    import hashlib
    import json
    with open(os.path.join(ROOT, "tests", "golden", "walking_log_sha256.json")) as f:
        want = json.load(f)
    for k in ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub"):
        a = getattr(walking_log, k)
        assert list(a.shape) == want[k]["shape"], k
        assert hashlib.sha256(np.ascontiguousarray(a, dtype="<f8").tobytes()).hexdigest() == want[k]["sha256"], k


def test_synthetic_shapes():
    from fcc_qp_b200 import synthetic as syn
    dims = {"humanoid": (90, 48, 12, 66), "quadruped": (54, 30, 12, 30), "multicontact": (120, 66, 24, 72)}
    for name, (n, m, nc, lcs) in dims.items():       # SURVEY.md 8d
        qp = syn.make_batch(syn.SHAPES[name], 3)
        assert (qp.n, qp.m, qp.nc, qp.lambda_c_start) == (n, m, nc, lcs)
        assert np.array_equal(qp.Q, qp.Q.transpose(0, 2, 1))
        assert np.linalg.matrix_rank(qp.A_eq[0]) == m
        again = syn.make_batch(syn.SHAPES[name], 3)
        assert np.array_equal(qp.A_eq, again.A_eq) and np.array_equal(qp.b, again.b)


def test_roofline_arithmetic():
    import bench
    # SURVEY.md 8d: Cassie 48,816 B in + 520 B out
    assert bench.algorithmic_bytes_per_qp(60, 38, 12) == 48816 + 520
    assert abs(bench.algorithmic_flops_per_qp(60, 38, 1, cold=False) - (98 ** 3 / 3 + 2 * 98 ** 2)) < 1e-6


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: every array GetSolution() returns, as float64 .npy, under the API's names."""
    import torch
    import bench
    from fcc_qp_b200.batch import BatchDetails, BatchSolution
    rng = np.random.default_rng(0)
    z = torch.from_numpy(rng.standard_normal((5, 4)))
    vec = lambda: torch.from_numpy(rng.random(5))
    it, st = torch.tensor([0, 3, 100, 7, 0], dtype=torch.int32), torch.tensor([0, 0, 1, 0, 2], dtype=torch.int32)
    sol = BatchSolution(BatchDetails(it, vec(), vec(), vec(), vec(), st), z)
    bench.dump_outputs(str(tmp_path / "out"), sol)
    want = {"z": z, "n_iter": it, "solve_status": st, "eps_bounds": sol.details.eps_bounds,
            "eps_friction_cone": sol.details.eps_friction_cone, "bounds_viol": sol.details.bounds_viol,
            "friction_cone_viol": sol.details.friction_cone_viol}
    assert sorted(p.name for p in (tmp_path / "out").iterdir()) == sorted(k + ".npy" for k in want)
    for k, v in want.items():
        got = np.load(tmp_path / "out" / (k + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got, v.numpy()), k


def test_cpp_dropin_compiles_against_eigen_surface():
    """A C++ caller of the reference's Eigen-typed FCCQP surface (src/fcc_qp.hpp:73-121) compiles and
    links against include/fcc_qp.hpp + libfccqp_b200.so unchanged (tests/cpp/dropin_main.cpp).
    Needs Eigen headers: the reference's vendored copy, present in the build container only."""
    import os
    from fcc_qp_b200 import build
    if not os.path.isdir("/root/reference/eigen"):
        pytest.skip("no Eigen headers here")
    tgt = build.build_cpp_dropin(force=True)
    assert tgt and os.path.exists(tgt)


def test_pybind_batch_class_is_bound_and_has_no_cpu_path():
    """fcc_qp::FCCQPBatch through the pybind11 module: the binding parses numpy stacks and DLPack tensors on the
    host side; without a CUDA device the host path fails loudly and a CPU tensor is refused before any launch."""
    import numpy as np
    import torch
    from fcc_qp_b200 import fcc_qp_solver as mod
    s = mod.FCCQPBatch(6, 3, 0, 0)
    for name in ("Solve", "SolveDLPack", "GetSolution", "set_options", "set_warm_start", "set_rho", "set_max_iter",
                 "set_structure", "contact_vars_start"):
        assert hasattr(s, name), name
    z = lambda *shape: torch.zeros(shape, dtype=torch.float64)
    outs = (z(2, 6), z(2, 6), z(2, 0), torch.zeros(2, dtype=torch.int32), torch.zeros(2, dtype=torch.int32), z(4, 2))
    with pytest.raises(TypeError, match="CUDA device memory"):
        s.SolveDLPack(z(2, 6, 6), z(2, 6), z(2, 3, 6), z(2, 3), z(0), z(6), z(6), *outs)
    with pytest.raises(ValueError):
        s.Solve(np.zeros((2, 6, 6)), np.zeros((2, 5)), np.zeros((2, 3, 6)), np.zeros((2, 3)), np.zeros(0), np.zeros(6), np.zeros(6))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            s.Solve(np.zeros((2, 6, 6)), np.zeros((2, 6)), np.zeros((2, 3, 6)), np.zeros((2, 3)), np.zeros(0), np.zeros(6), np.zeros(6))


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The ctypes mirrors of the C-ABI descriptors (fcc_qp_b200/_native.py) against what a C compiler makes of include/fccqp.h:
    sizes and the offsets of the last members."""
    import subprocess
    import ctypes as C
    from fcc_qp_b200 import _native as nat
    src = tmp_path / "abi.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "fccqp.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(fccqp_options), sizeof(fccqp_details), sizeof(fccqp_batch_desc),
         offsetof(fccqp_batch_desc, struct_caps), sizeof(fccqp_wbc_desc), sizeof(fccqp_polish_desc),
         offsetof(fccqp_polish_desc, polished), offsetof(fccqp_polish_desc, eps_objective));
  printf("%d %d %d %d %d\n", FCCQP_ABI_VERSION, FCCQP_PRECISION_FP32, FCCQP_STRUCTURE_REFINE, FCCQP_SCHEDULE_LPT, FCCQP_STATUS_NUMERICAL_ISSUE);
  return 0;
}
''')
    exe = tmp_path / "abi"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    l1, l2 = subprocess.check_output([str(exe)], text=True).splitlines()
    got = [int(v) for v in l1.split()]
    want = [C.sizeof(nat.Options), C.sizeof(nat.Details), C.sizeof(nat.BatchDesc), nat.BatchDesc.struct_caps.offset,
            C.sizeof(nat.WbcDesc), C.sizeof(nat.PolishDesc), nat.PolishDesc.polished.offset, nat.PolishDesc.eps_objective.offset]
    assert got == want, (got, want)
    assert [int(v) for v in l2.split()] == [nat.ABI_VERSION, 2, nat.STRUCTURE_REFINE, nat.SCHEDULE_LPT, nat.STATUS_NUMERICAL_ISSUE]
