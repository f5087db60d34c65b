"""Warp-per-QP kernel (fccqp_warp.cuh): the mapping for problems with n + m <= 32.  Checked against the C restatement of
the reference on random small QPs (cold, warm sequences, over-relaxation), against the CTA-per-QP kernels on the same
inputs (FCCQP_NO_WARP=1), and with the long-running-QP operator switched on from the first iteration / never."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from kernel_layout import layout_bytes
from test_gpu_random_shapes import random_qps, rel

pytestmark = pytest.mark.gpu
OPTS = dict(max_iter=200, rho=1e-3, eps_fcone=1e-7, eps_bound=1e-7)
# n + m = 32 is the largest shape of the warp kernel, 33 the smallest of the CTA-per-QP kernels
SMALL = [(5, 2, 3, 1), (12, 6, 6, 3), (18, 14, 6, 10), (24, 8, 9, 0), (32, 0, 12, 20), (3, 0, 3, 0), (20, 12, 0, 0),
         (27, 6, 9, 12)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def solver(n, m, nc, lcs, **kw):
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    s = FCCQPBatch(n, m, nc, lcs)
    s.set_options(FCCQPOptionsB(**{**OPTS, **kw}))
    return s


@pytest.mark.parametrize("n,m,nc,lcs", SMALL)
def test_small_shapes_cold_and_warm_match_the_restatement(n, m, nc, lcs):
    from fcc_qp_b200 import _native as nat
    rng = np.random.default_rng(77 * n + m)
    B = 1024
    qp = random_qps(rng, B, n, m, nc, lcs)
    ref = oracle.Oracle("port").solve_batch(qp, warm_mode=0, nthreads=8, **OPTS)
    s = solver(n, m, nc, lcs)
    s.Solve(qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)
    sol = s.GetSolution()
    smem = 4 * (n + m) * ((n + m) | 1) * 8 if n + m <= 32 else layout_bytes(n, m, nc)   # else the general kernel
    assert nat.last_launch_info()["block"] == 128 and nat.last_launch_info()["smem_bytes"] == smem
    same = sol.details.n_iter == ref["n_iter"]
    assert rel(sol.z[same], ref["z"][same]) <= 1e-6
    assert (~same).mean() <= 0.01, (~same).sum()
    assert np.array_equal(sol.details.solve_status[same], ref["status"][same])
    assert np.abs(sol.details.eps_bounds - ref["res_bounds"])[same].max() <= 1e-6
    assert np.abs(sol.details.friction_cone_viol - ref["fcone_viol"])[same].max() <= 1e-6
    # lane-wise warm start: the same lanes walk on to perturbed QPs with carried state
    lanes = oracle.Oracle("port").lanes(64, n, m, nc, lcs)
    lanes.set_options(**OPTS)
    w = solver(n, m, nc, lcs)
    sub = qp.take(np.arange(64))
    for t in range(4):
        r = lanes.solve(sub, warm=t > 0)
        w.set_warm_start(t > 0)
        w.Solve(sub.Q, sub.b, sub.A_eq, sub.b_eq, sub.friction_coeffs, sub.lb, sub.ub)
        g = w.GetSolution()
        ok = g.details.n_iter == r["n_iter"]
        assert ok.mean() >= 0.95 and rel(g.z[ok], r["z"][ok]) <= 1e-6, t
        sub = qp.take(np.arange(64) + 64 * (t + 1))


def test_relaxation_on_the_warp_kernel():
    n, m, nc, lcs = 12, 6, 6, 3
    qp = random_qps(np.random.default_rng(5), 256, n, m, nc, lcs)
    port = oracle.Oracle("port")
    port.set_relaxation(1.5)
    try:
        ref = port.solve_batch(qp, warm_mode=0, nthreads=4, **OPTS)
    finally:
        port.set_relaxation(1.0)
    s = solver(n, m, nc, lcs, relaxation=1.5)
    s.Solve(qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)
    sol = s.GetSolution()
    same = sol.details.n_iter == ref["n_iter"]
    assert same.mean() >= 0.98 and rel(sol.z[same], ref["z"][same]) <= 1e-6


@pytest.mark.parametrize("env", [{"FCCQP_NO_WARP": "1"}, {"FCCQP_FULL_INVERSE_AT": "1"}, {"FCCQP_FULL_INVERSE_AT": "1000000"}])
def test_warp_kernel_agrees_with_the_cta_kernels_and_across_operator_switch(env, tmp_path):
    """Same inputs through (a) the CTA-per-QP kernels, (b) the warp kernel with every iterating QP on the explicit operator
    from its first real x-update, (c) never: all within 1e-8 of the default configuration, identical counts."""
    code = r'''
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from test_gpu_random_shapes import random_qps
from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
out = {}
for n, m, nc, lcs in [(12, 6, 6, 3), (24, 8, 9, 0), (30, 2, 12, 10)]:
    qp = random_qps(np.random.default_rng(n), 512, n, m, nc, lcs)
    s = FCCQPBatch(n, m, nc, lcs); s.set_options(FCCQPOptionsB(max_iter=200, rho=1e-3, eps_fcone=1e-7, eps_bound=1e-7))
    s.Solve(qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)
    r = s.GetSolution()
    out[f"z{n}"] = r.z; out[f"it{n}"] = r.details.n_iter
np.savez(sys.argv[2], **out)
'''
    a, b = str(tmp_path / "a.npz"), str(tmp_path / "b.npz")
    base = {k: v for k, v in os.environ.items() if k not in ("FCCQP_NO_WARP", "FCCQP_FULL_INVERSE_AT")}
    for path, e in ((a, base), (b, dict(base, **env))):
        r = subprocess.run([sys.executable, "-c", code, ROOT, path], env=e, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
    A, Bz = np.load(a), np.load(b)
    for n in (12, 24, 30):
        same = A[f"it{n}"] == Bz[f"it{n}"]
        assert same.mean() >= 0.99, (env, n, (~same).sum())
        assert rel(A[f"z{n}"][same], Bz[f"z{n}"][same]) <= 1e-8, (env, n)


def test_dropin_object_on_small_problems_takes_the_warp_kernel():
    """The single-problem FCCQP object (pybind, host arrays) on the reference-generated known answers: projection of a
    point onto one friction cone (n = 3) and the closed-form equality-constrained QP (n = 12, m = 5, n_iter = 0)."""
    from fcc_qp import FCCQP, FCCQPOptions
    from fcc_qp_b200 import _native as nat
    kats = np.load(os.path.join(ROOT, "tests", "golden", "kats.npz"))
    o = FCCQPOptions(); o.max_iter, o.rho, o.eps_fcone, o.eps_bound = 2000, 1.0, 1e-10, 1e-10
    inf3 = np.full(3, np.inf)
    for f, z in zip(kats["cone_f"], kats["cone_z"]):
        s = FCCQP(3, 0, 3, 0); s.set_options(o)
        s.Solve(np.eye(3), -f, np.zeros((0, 3)), np.zeros(0), [0.5], -inf3, inf3)
        assert nat.last_launch_info()["block"] == 128 and nat.last_launch_info()["smem_bytes"] == 4 * 3 * 3 * 8
        assert np.abs(s.GetSolution().z - z).max() <= 1e-8
    o2 = FCCQPOptions(); o2.max_iter, o2.rho, o2.eps_fcone, o2.eps_bound = 100, 1e-3, 1e-6, 1e-6
    s = FCCQP(12, 5, 0, 0); s.set_options(o2)
    inf12 = np.full(12, np.inf)
    s.Solve(kats["eq_Q"], kats["eq_b"], kats["eq_A"], kats["eq_beq"], [], -inf12, inf12)
    r = s.GetSolution()
    assert r.details.n_iter == int(kats["eq_n_iter"]) == 0
    assert np.abs(r.z - kats["eq_z"]).max() <= 1e-9 * max(1.0, np.abs(kats["eq_z"]).max())
    # warm restart of the same object (carried state on the device)
    s.set_warm_start(True)
    s.Solve(kats["eq_Q"], kats["eq_b"], kats["eq_A"], kats["eq_beq"], [], -inf12, inf12)
    assert np.abs(s.GetSolution().z - kats["eq_z"]).max() <= 1e-9 * max(1.0, np.abs(kats["eq_z"]).max())


@pytest.mark.parametrize("n,m,nc,lcs", [(6, 3, 3, 3), (12, 6, 6, 3), (24, 8, 6, 0), (32, 0, 12, 20)])
def test_fp32_arithmetic_mode_within_its_stated_bound(n, m, nc, lcs):
    """FCCQP_PRECISION_FP32 (include/fccqp.h): float32 problem data and FP32 arithmetic on the warp kernel.  Stated bound:
    1e-4 relative on z and on the objective against the FP64 reference (here: its pinned C restatement on the ORIGINAL
    double data) for QPs whose rho-KKT matrix has cond <= 1e3, eps >= 1e-4; same status.  Checked on the random set
    (cond <= 80) and on the same QPs with the rows of A_eq scaled apart (cond up to ~1e3: QPs beyond are left out)."""
    from fcc_qp_b200 import _native as nat
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    from fcc_qp_b200.synthetic import scale_constraint_rows
    opts = dict(max_iter=200, rho=1e-3, eps_fcone=1e-4, eps_bound=1e-4)
    base = random_qps(np.random.default_rng(31 * n + m), 512, n, m, nc, lcs)
    sets = [base] + ([scale_constraint_rows(base, np.random.default_rng(3), 1.0)] if m else [])
    for qp in sets:
        cond = np.empty(qp.batch)
        for i in range(qp.batch):
            K = np.zeros((n + m, n + m))
            K[:n, :n] = qp.Q[i] + opts["rho"] * np.eye(n); K[n:, :n] = qp.A_eq[i]; K[:n, n:] = qp.A_eq[i].T
            cond[i] = np.linalg.cond(K)
        ok = cond <= 1e3
        assert ok.mean() > 0.5
        ref = oracle.Oracle("port").solve_batch(qp, warm_mode=0, nthreads=8, **opts)
        s = FCCQPBatch(n, m, nc, lcs, precision="fp32"); s.set_options(FCCQPOptionsB(**opts))
        s.Solve(qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)
        sol = s.GetSolution()
        assert nat.last_launch_info()["smem_bytes"] == 4 * (n + m) * ((n + m) | 1) * 4      # float slabs: the FP32 instance ran
        err = np.abs(sol.z - ref["z"]).max(axis=1) / np.maximum(1.0, np.abs(ref["z"]).max(axis=1))
        assert err[ok].max() <= 1e-4, err[ok].max()
        obj = lambda z: 0.5 * np.einsum("bi,bij,bj->b", z, qp.Q, z) + np.einsum("bi,bi->b", qp.b, z)
        oerr = np.abs(obj(sol.z) - obj(ref["z"])) / np.maximum(1.0, np.abs(obj(ref["z"])))
        assert oerr[ok].max() <= 1e-4, oerr[ok].max()
        assert np.array_equal(sol.details.solve_status[ok], ref["status"][ok])
        assert (sol.details.n_iter[ok] == ref["n_iter"][ok]).mean() >= 0.98


def test_fp32_mode_on_a_large_problem_runs_as_fp32_data(walking_log):
    """n + m > 32: no FP32-arithmetic kernel; FCCQP_PRECISION_FP32 then means float32 data with FP64 arithmetic, bit for bit
    the result of FCCQP_PRECISION_FP32_DATA."""
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    qp = walking_log.take(np.arange(64))
    out = []
    for prec in ("fp32", "fp32_data"):
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start, precision=prec)
        s.set_options(FCCQPOptionsB(100, 5e-5, 1e-6, 1e-6))
        s.Solve(qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)
        out.append(s.GetSolution())
    assert np.array_equal(out[0].z, out[1].z) and np.array_equal(out[0].details.n_iter, out[1].details.n_iter)
