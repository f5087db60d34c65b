"""Every compiled solve-kernel instance at the shapes that select it, against the C restatement of the reference run live on
the same inputs.

The launchers (fcc_qp_b200/csrc/fccqp_capi.cu) pick the instance from the problem shape: the structure-exploiting kernel
takes 64 / 96 / 128 / 256 threads from need = max(n, padded reduced KKT size) with cuts at 64, 96 and 128, its probe
takes 256 threads when n > 128, an odd n switches its classification scan to one thread per column and per-element
copies, and the general kernel takes 256 threads above 128 padded KKT rows.  The parity sets elsewhere stop at
need = 120 with even n, so each cell here asserts which instance ran (fccqp_last_launch_info, fccqp_last_struct_info)
and then holds it to the parity bar of test_gpu_parity.py:

* z and the objective within 1e-6 relative on lanes whose iteration count matches the restatement's;
* identical counts on at least 99.5 % of the lanes, every difference explained by its exit margin;
* identical status where the counts agree;
* and the batch must exercise the iteration: at least 5 % of the lanes iterate, some past iteration 6, where long-running
  QPs switch to the compact operator loop.

The last cells find the largest problem the device accepts and check that it is the one include/fccqp.h states.
"""
import os
import re
import types

import numpy as np
import pytest

import oracle
from conftest import LOG_OPTS
from fcc_qp_b200 import synthetic as syn
from kernel_layout import layout_bytes, up8
from test_gpu_option_paths import cold_ref, dev, oracle_with, run, solver
from test_gpu_parity import explain_count_mismatches, rel_err
from test_gpu_split import check_split, column_major, strided

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = 256
RANDOM_OPTS = dict(max_iter=200, rho=1e-3, eps_fcone=1e-7, eps_bound=1e-7)


# Whole-body-control shapes for the structure-exploiting kernel: nr = nv, ndp = nc, nd0 = nh, so the reduced KKT system
# has up8(nv) + up8(m) + up8(nh) rows.  (nv, nu, nh, nc, threads, make_batch tuning): need 64 / 65 (odd), 96 / 97 (odd),
# 128 / 129 (odd), and the largest accepted problem (n = 140, m = 76, 224 padded rows).  The larger shapes bind more
# cones at the default tuning and would run most lanes to max_iter: smaller joint columns and task commands there.
TUNED = dict(joint_scale=0.02, ydd_sigma=0.3)
WBC = {
    "need64": (22, 18, 0, 12, 64, {}),
    "need65-odd": (22, 19, 0, 12, 96, {}),
    "need96": (30, 24, 0, 21, 96, TUNED),
    "need97-odd": (30, 22, 3, 21, 128, TUNED),
    "need128": (40, 34, 0, 27, 128, TUNED),
    "need129-odd": (40, 35, 0, 27, 256, TUNED),
    "limit": (48, 40, 4, 24, 256, TUNED),
}


def wbc(name, batch=B, seed=None):
    nv, nu, nh, nc, threads, kw = WBC[name]
    kw = dict(kw)
    shape = syn.Shape(name, nv, nu, nh, nc, seed=1000 + nv + nu + nh + nc, joint_scale=kw.pop("joint_scale", 0.05))
    qp = syn.make_batch(shape, batch, seed=seed, **kw)
    return qp, threads, (nv, nc, nh), up8(nv) + up8(qp.m) + up8(nh)


def assert_bar(qp, r, ref, opts, state=None, z_tol=1e-6, what=""):
    it, z = r.n_iter, r.z
    assert (ref["n_iter"] > 0).mean() >= 0.05 and (ref["n_iter"] > 6).any(), (what, "batch does not iterate")
    same = it == ref["n_iter"]
    assert same.mean() >= 0.995, (what, int((~same).sum()))
    err = rel_err(z[same], ref["z"][same])
    assert err.max() <= z_tol, (what, err.max())
    o, oref = qp.objective(z), qp.objective(ref["z"])
    assert (np.abs(o - oref) / np.maximum(1.0, np.abs(oref)))[same].max() <= 1e-6, what
    assert np.array_equal(r.status[same], ref["status"][same]), what
    margins = explain_count_mismatches(qp, it, ref["n_iter"], opts=opts, state=state, z_gpu=z)
    print(f"{what}: iterating {(ref['n_iter'] > 0).mean():.2f}, past 6 {int((ref['n_iter'] > 6).sum())}, "
          f"max err {err.max():.2e}, count differences {len(margins)}")


def assert_struct_ran(r, threads, caps, rows, deferred=0):
    from fcc_qp_b200 import _native as nat
    info = nat.last_struct_info()
    assert r.struct_used and r.launch["block"] == threads, (r.launch, info)
    assert tuple(info["caps"]) == caps and info["rows"] == rows and info["deferred"] == deferred, info


# ---- 1. structure-exploiting kernel at each thread-count cut (and the 256-thread instance at the limit): cold, then
# one warm step from the carried state
@pytest.mark.parametrize("name", list(WBC))
def test_struct_instance_cold_and_warm(name):
    qp, threads, caps, rows = wbc(name)
    qp2 = syn.random_walk(qp, np.random.default_rng(11))
    with oracle_with() as o:
        lanes = o.lanes(qp.batch, qp.n, qp.m, qp.nc, qp.lambda_c_start)
        lanes.set_options(**LOG_OPTS)
        ref0, ref1 = lanes.solve(qp, warm=False), lanes.solve(qp2, warm=True)
    s = solver(qp, LOG_OPTS, structure="probe")
    r0 = run(s, qp)
    assert r0.launches == 3                        # probe, structure-exploiting kernel, general kernel (nothing deferred)
    assert_struct_ran(r0, threads, caps, rows)
    assert_bar(qp, r0, ref0, LOG_OPTS, what=f"{name} cold")
    state = tuple(a.cpu().numpy().copy() for a in s.GetState())
    r1 = run(s, qp2, warm=True)
    assert_struct_ran(r1, threads, caps, rows)
    assert_bar(qp2, r1, ref1, LOG_OPTS, state=state, what=f"{name} warm")


# The classification must read any nonzero off-diagonal entry as coupling, whatever its sign: one torque and one slack
# variable of every QP are tied by the PSD block c [[1, -1], [-1, 1]], so both leave the separable classes.
@pytest.mark.parametrize("name", ["need64", "need65-odd", "need97-odd", "need129-odd"])
def test_negative_coupling_keeps_variables_in_the_kkt_system(name):
    qp, threads, (nr, ndp, nd0), _ = wbc(name)
    nv, nu, nh = WBC[name][:3]
    u, e, c = nv, qp.n - 1, 1e-3
    qp.Q[:, [u, e], [u, e]] += c
    qp.Q[:, u, e] -= c
    qp.Q[:, e, u] -= c
    ref = cold_ref(qp, LOG_OPTS)
    r = run(solver(qp, LOG_OPTS, structure="probe"), qp)
    rows = up8(nr + 2) + up8(qp.m) + up8(nd0)
    assert_struct_ran(r, threads, (nr + 2, ndp, nd0), rows)
    assert_bar(qp, r, ref, LOG_OPTS, what=f"{name} negative coupling")


# ---- 2. the 256-thread structure-exploiting instance under every option and layout, at n > 128 and at the size limit;
# the adaptive-rho instances of the 64-, 96- and 128-thread kernels
CELLS_256 = ["adapt5", "relax1.6", "refine", "strided", "caps-too-small", "host-classify"]


@pytest.mark.parametrize("name,cell", [(name, cell) for name in ("need129-odd", "limit") for cell in CELLS_256] +
                         [(name, "adapt5") for name in ("need64", "need65-odd", "need97-odd", "need128")])
def test_struct_option_cells(name, cell):
    qp, threads, caps, rows = wbc(name)
    opt = {"adapt5": dict(adapt_rho_interval=5), "relax1.6": dict(relaxation=1.6)}.get(cell, {})
    with oracle_with(**opt) as o:
        ref = o.solve_batch(qp, warm_mode=0, nthreads=8, **LOG_OPTS)
        if cell == "host-classify":
            # host arrays: the host-side twin of the classification sizes the kernel; it must agree with the probe
            from fcc_qp_b200 import _native as nat
            s = solver(qp, LOG_OPTS, structure="auto")
            s.Solve(qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)
            sol = s.GetSolution()
            info = nat.last_struct_info()
            assert info["used"] and tuple(info["caps"]) == caps and info["rows"] == rows and info["deferred"] == 0, info
            assert nat.last_launch_info()["block"] == threads
            host = types.SimpleNamespace(z=sol.z, n_iter=sol.details.n_iter, status=sol.details.solve_status)
            assert_bar(qp, host, ref, LOG_OPTS, what=f"{name} host path")
            return
        s = solver(qp, LOG_OPTS, structure=(8, 4, 2) if cell == "caps-too-small" else "probe", **opt)
        s.refine = cell == "refine"
        Q, A = (strided(dev(qp.Q)), column_major(dev(qp.A_eq))) if cell == "strided" else (None, None)
        r = run(s, qp, Q, A)
        if cell == "caps-too-small":
            # every QP exceeds the caps and is handed to the general kernel's 256-thread instance
            assert_struct_ran(r, threads, (8, 4, 2), 8 + up8(qp.m) + 8, deferred=qp.batch)
        else:
            assert_struct_ran(r, threads, caps, rows)
        # the refined reduced pre-solve is as close as the general kernel's (test_gpu_structure.py)
        assert_bar(qp, r, ref, LOG_OPTS, z_tol=5e-9 if cell == "refine" else 1e-6, what=f"{name} {cell}")


# ---- 3. two-stage cold solve (first-stage kernel, then the resume launch): bit-identical to the single launch that
# batches below the threshold take.  Every variant on the 256-thread instance; the refining first stage also at 64 and
# 128 threads (the walking-log split tests cover 96 threads, and the plain first stage at 64 and 128).
@pytest.mark.parametrize("name,variant", [("limit", "plain"), ("limit", "refine"), ("limit", "schedule-from-previous"),
                                          ("need64", "refine"), ("need128", "refine")])
def test_struct_two_stage_matches_single_launch(name, variant):
    import torch
    qp, threads, caps, rows = wbc(name, batch=64)
    r = run(solver(qp, LOG_OPTS, structure="probe"), qp)
    assert_struct_ran(r, threads, caps, rows)   # the first stage takes the thread count of the full kernel
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    big = 8 * r.launch["ctas_per_sm"] * sms + 37   # at the threshold of the two-stage solve, not a multiple of 128
    qp, *_ = wbc(name, batch=big, seed=5)
    # (check_split asserts four launches per solve: probe, first stage, resume, general)
    out, info = check_split(qp, refine=variant == "refine", lpt=variant == "schedule-from-previous")
    assert info["used"] and tuple(info["caps"]) == caps and info["rows"] == rows and info["deferred"] == 0, info
    assert (out["n_iter"] > 0).mean() >= 0.05 and (out["n_iter"] > 6).any()


# ---- 4. general kernel: 128 / 256 threads at 128 and 136 padded rows, 256 at the largest accepted size; FP64 and
# float32 data, each with and without adaptive rho (the four instances of solve_instance per thread count)
@pytest.mark.parametrize("n,m,nc,lcs", [(72, 50, 12, 30), (80, 50, 12, 7), (120, 100, 15, 101)],
                         ids=["N8=128", "N8=136", "N8=224"])
@pytest.mark.parametrize("precision", ["fp64", "fp32_data"])
@pytest.mark.parametrize("adapt", [0, 5])
def test_general_instance(n, m, nc, lcs, precision, adapt):
    import dataclasses
    qp = syn.random_qps(np.random.default_rng(n + m + adapt), B, n, m, nc, lcs)
    if precision == "fp32_data":   # the reference is the FP64 restatement on the float32-rounded inputs
        r32 = lambda a: np.ascontiguousarray(a.astype(np.float32).astype(np.float64))
        qp = dataclasses.replace(qp, Q=r32(qp.Q), b=r32(qp.b), A_eq=r32(qp.A_eq), b_eq=r32(qp.b_eq),
                                 friction_coeffs=r32(qp.friction_coeffs), lb=r32(qp.lb), ub=r32(qp.ub))
    opt = dict(adapt_rho_interval=adapt)
    with oracle_with(**opt) as o:
        ref = o.solve_batch(qp, warm_mode=0, nthreads=8, **RANDOM_OPTS)
        r = run(solver(qp, RANDOM_OPTS, structure="dense", precision=precision, **opt), qp)
        assert r.launches == 1 and not r.struct_used
        N8 = up8(n) + up8(m)
        assert r.launch["block"] == (128 if N8 <= 128 else 256) and r.launch["smem_bytes"] == layout_bytes(n, m, nc), r.launch
        assert_bar(qp, r, ref, RANDOM_OPTS, what=f"general N8={N8} {precision} adapt={adapt}")


# ---- 5. the size limit
def stated_limit():
    """Largest padded n + m that include/fccqp.h and INTEGRATION.md state."""
    found = []
    for doc in ("include/fccqp.h", "INTEGRATION.md"):
        with open(os.path.join(ROOT, doc)) as f:
            found += [int(v) for v in re.findall(r"padded n \+ m (?:<=|≤) (\d+)", f.read())]
    assert found and len(set(found)) == 1, found
    return found[0]


def accepted(n, m, nc):
    from fcc_qp import FCCQP
    try:
        FCCQP(n, m, nc, 0)
    except RuntimeError as e:
        assert "shared memory" in str(e), e
        return False
    return True


def test_size_limit_is_the_stated_one():
    """The largest padded KKT size (n and m each rounded up to a multiple of 8) that the single-problem object accepts,
    over every split with m8 <= n8 and several contact counts, is the same for all of them and is the documented one."""
    limits = set()
    for N8 in range(192, 265, 8):
        ok = {accepted(n8 - d, N8 - n8 - e, nc) for n8 in range(up8((N8 + 1) // 2), N8, 8)
              for d, e in ((0, 0), (7, 3)) for nc in (0, 3 * ((n8 - d) // 3))}
        assert len(ok) == 1, N8          # the limit does not depend on the split
        limits.add((N8, ok.pop()))
    largest = max(N8 for N8, ok in limits if ok)
    assert all(ok == (N8 <= largest) for N8, ok in limits)
    assert largest == stated_limit()


def test_largest_problem_solves_and_next_size_is_refused():
    """The limit shape of the structure-exploiting cells is at the stated limit; one tile row more (n = 144, m = 81) is
    refused with FCCQP_E_UNSUPPORTED on the host and device batch paths and by the single-problem object."""
    from fcc_qp_b200 import FCCQPError
    qp, *_ = wbc("limit", batch=4)
    assert up8(qp.n) + up8(qp.m) == stated_limit()
    r = run(solver(qp, LOG_OPTS, structure="dense"), qp)   # the general kernel at its smallest occupancy
    assert r.launch["block"] == 256 and r.launch["ctas_per_sm"] == 1 and r.launch["smem_bytes"] == layout_bytes(qp.n, qp.m, qp.nc)
    ref = oracle.Oracle("port").solve_batch(qp, warm_mode=0, **LOG_OPTS)
    assert rel_err(r.z, ref["z"]).max() <= 1e-6 and np.array_equal(r.n_iter, ref["n_iter"])
    n = 144
    m = stated_limit() + 8 - n - 7
    big = syn.random_qps(np.random.default_rng(1), 2, n, m, 0, 0)
    args = (big.Q, big.b, big.A_eq, big.b_eq, np.zeros(0), big.lb, big.ub)
    for path in ("host", "device"):
        s = solver(big, LOG_OPTS)
        with pytest.raises(FCCQPError) as e:
            s.Solve(*(args if path == "host" else [dev(a) for a in args]))
        assert e.value.code == -3, path
    assert not accepted(n, m, 0)
