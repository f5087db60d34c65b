"""Per-lane rho (fccqp_batch_solve_rho, FCCQPBatch.set_rho(array)), path by path.

1. A uniform-valued array (every entry options.rho) equals the call without it: such calls run the instances that keep rho
   per QP (those of adaptive rho), so the bar is identical counts and status and z within 1e-12 relative; the array comes
   back unchanged.
2. Distinct per-lane rho: every lane equals the uniform call at its rho (same bar), and one reference object per lane
   after set_rho(rho_i) under the parity bar of test_gpu_parity.py.
3. Adaptive rho every 5 iterations over a warm sequence with the carried array: the C restatement driven lane by lane
   with set_rho(last_rho) before every step, under the bar of test_adaptive_rho.py; the returned rho is the restatement's.
4. A warm_lanes mask with per-lane rho: every lane equals the uniform call of its kind at its rho.
5. CUDA graph: replays carry rho from step to step, and an entry changed in place between replays takes effect.
6. Entries that are not finite or not > 0 end their lane with NUMERICAL_ISSUE and n_iter 0 and stay as they were, in
   cold, warm and mixed calls.
7. FCCQP_SCHEDULE_LPT with an array changes the processing order only.
"""
import numpy as np
import pytest

import oracle
import rho_oracle
from conftest import LOG_OPTS
from fcc_qp_b200 import synthetic as syn
from test_gpu_parity import Z_TOL, explain_count_mismatches, rel_err
from test_gpu_warm_lanes import FP32_OPTS, RANDOM_OPTS, scattered_mask, shared_set, solver_factory

pytestmark = pytest.mark.gpu
RHOS = np.array([1e-6, 5e-5, 1e-3, 1e-1])
KEYS = ("z", "mu_x", "mu_c", "n_iter", "status", "res_b", "res_f", "bviol", "fviol")


def _np(a):
    return a.cpu().numpy().copy() if hasattr(a, "cpu") else np.array(a, copy=True)


def solve_step(make, qp0, qp1, warm=True, rho=None, device=True, Q=None, A=None):
    """A fresh solver (or `s`): a cold solve of qp0 at options.rho (the carried state), then one solve of qp1 with
    set_warm_start(warm) and, when given, set_rho(rho) -- a float, or a copy of a per-lane array.  Returns its outputs and
    the array after the call."""
    import torch
    s = make()
    f32 = s.precision != "fp64"
    dt = torch.float32 if f32 else torch.float64
    t = lambda a: torch.as_tensor(a, dtype=dt, device="cuda:0")

    def args(qp):
        if not device:
            return [qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub]
        return [t(qp.Q) if Q is None else Q, t(qp.b), t(qp.A_eq) if A is None else A, t(qp.b_eq), t(qp.friction_coeffs),
                t(qp.lb), t(qp.ub)]

    s.set_warm_start(False)
    s.Solve(*args(qp0))
    if isinstance(warm, np.ndarray) and device:
        warm = torch.as_tensor(warm, device="cuda:0")
    s.set_warm_start(warm)
    if isinstance(rho, float):
        s.set_rho(rho)
    elif rho is not None:
        s.set_rho(torch.as_tensor(rho, dtype=torch.float64, device="cuda:0").clone() if device else np.array(rho, np.float64))
    s.Solve(*args(qp1))
    torch.cuda.synchronize()
    sol, d = s.GetSolution(), s.GetSolution().details
    x, mux, muc = s.GetState()
    out = dict(z=sol.z, mu_x=mux, mu_c=muc, n_iter=d.n_iter, status=d.solve_status, res_b=d.eps_bounds,
               res_f=d.eps_friction_cone, bviol=d.bounds_viol, fviol=d.friction_cone_viol)
    out = {k: _np(v) for k, v in out.items()}
    out["rho"] = None if s.rho_lanes is None else _np(s.rho_lanes)
    return out


def assert_close(got, want, lanes, what, ztol=1e-12):
    """Identical counts and status, z (and the duals) within ztol relative: the bar between a call that runs an instance
    keeping rho per QP and one that does not (bit-identical where both run the same instance)."""
    assert np.array_equal(got["n_iter"][lanes], want["n_iter"][lanes]), (what, int((got["n_iter"] != want["n_iter"])[lanes].sum()))
    assert np.array_equal(got["status"][lanes], want["status"][lanes]), what
    for k in ("z", "mu_x"):
        assert rel_err(got[k][lanes], want[k][lanes]).max() <= ztol, (what, k, rel_err(got[k][lanes], want[k][lanes]).max())


def assert_equal(got, want, lanes, what):
    for k in KEYS:
        assert got[k][lanes].tobytes() == want[k][lanes].tobytes(), (what, k)


@pytest.fixture(scope="module")
def log512(walking_log):
    qp0 = walking_log.take(np.arange(512) * 3)
    return qp0, syn.random_walk(qp0, np.random.default_rng(41))


@pytest.fixture(scope="module")
def log16k(walking_log):
    qp0 = walking_log.tile(16384)
    return qp0, syn.random_walk(qp0, np.random.default_rng(42))


def path_case(path, walking_log, log512, log16k):
    """(make, qp0, qp1, kwargs of solve_step) of one kernel path."""
    if path in ("warp-fp64", "warp-fp32"):
        qp0 = syn.random_qps(np.random.default_rng(43), 2048, 14, 5, 6, 6)
        prec = path.split("-")[1]
        return solver_factory(qp0, FP32_OPTS if prec == "fp32" else RANDOM_OPTS, precision=prec), qp0, \
            syn.random_walk(qp0, np.random.default_rng(44)), {}
    if path == "general":
        return solver_factory(log512[0], LOG_OPTS, structure="dense"), *log512, {}
    if path == "struct-single":
        return solver_factory(log512[0], LOG_OPTS, structure="probe"), *log512, {}
    if path == "struct-split":
        return solver_factory(log16k[0], LOG_OPTS, structure="probe"), *log16k, {}
    if path == "struct-fallback":
        return solver_factory(log16k[0], LOG_OPTS, structure=(8, 4, 2)), *log16k, {}
    if path == "host":
        qp0 = walking_log.tile(12288)
        return solver_factory(qp0, LOG_OPTS), qp0, syn.random_walk(qp0, np.random.default_rng(45)), dict(device=False)
    raise ValueError(path)


PATHS = ["warp-fp64", "warp-fp32", "general", "struct-single", "struct-split", "struct-fallback", "host"]


def lane_rhos(B, base):
    return np.where(np.arange(B) % 5 == 4, base, RHOS[np.arange(B) % 4])


@pytest.mark.parametrize("warm", [False, True])
@pytest.mark.parametrize("path", PATHS)
def test_uniform_and_distinct_rho(walking_log, log512, log16k, path, warm):
    """Cases 1 and 2 on one path, cold and warm."""
    make, qp0, qp1, kw = path_case(path, walking_log, log512, log16k)
    B = qp0.batch
    base = make().options.rho
    plain = solve_step(make, qp0, qp1, warm, **kw)
    uni = solve_step(make, qp0, qp1, warm, rho=np.full(B, base), **kw)
    assert_close(uni, plain, slice(None), f"{path} uniform")
    assert np.array_equal(uni["rho"], np.full(B, base))
    r = lane_rhos(B, base)
    got = solve_step(make, qp0, qp1, warm, rho=r, **kw)
    assert np.array_equal(got["rho"], r)                      # adaptive rho off: returned unchanged
    iterating = 0
    for v in np.unique(r):
        want = solve_step(make, qp0, qp1, warm, rho=float(v), **kw)
        assert_close(got, want, r == v, f"{path} rho {v}")
        iterating += int((want["n_iter"][r == v] > 0).sum())
    assert iterating > 0
    # the rho entries matter: lanes at 1e-6 and at 1e-1 iterate differently
    assert not np.array_equal(got["n_iter"], plain["n_iter"]) or got["z"].tobytes() != plain["z"].tobytes()


def test_uniform_and_distinct_rho_shared_structure():
    """Stride-0 Q / A_eq with an array runs the per-QP kernels (a cached factorization has one rho): it equals the same
    data with Q and A_eq materialised per QP, without the array (cold: the carried state of the two differs in its
    last bits)."""
    qp0, qp1, Q, A = shared_set()
    B = qp0.batch
    make = solver_factory(qp0, LOG_OPTS, structure="dense")   # (the general kernel on both sides)
    Qm, Am = Q.contiguous(), A.contiguous()
    for r in (np.full(B, LOG_OPTS["rho"]), lane_rhos(B, LOG_OPTS["rho"])):
        got = solve_step(make, qp0, qp1, False, rho=r, Q=Q, A=A)
        for v in np.unique(r):
            want = solve_step(make, qp0, qp1, False, rho=float(v), Q=Qm, A=Am)
            assert_close(got, want, r == v, f"shared rho {v}")
        assert np.array_equal(got["rho"], r)


def test_two_devices(walking_log):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    qp0 = walking_log.tile(24576)
    qp1 = syn.random_walk(qp0, np.random.default_rng(46))
    make = solver_factory(qp0, LOG_OPTS, device=[0, 1])
    r = lane_rhos(qp0.batch, LOG_OPTS["rho"])
    got = solve_step(make, qp0, qp1, True, rho=r, device=False)
    for v in np.unique(r):
        assert_close(got, solve_step(make, qp0, qp1, True, rho=float(v), device=False), r == v, f"two devices rho {v}")


@pytest.mark.parametrize("data", ["walking_log", "humanoid"])
def test_distinct_rho_matches_one_reference_object_per_lane(walking_log, data):
    """Cold solves, lane i against a reference object after set_rho(rho_i), under the parity bar of test_gpu_parity.py."""
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    B = 512
    qp = walking_log.take(np.arange(B) * 3) if data == "walking_log" else syn.make_batch(syn.HUMANOID, B, seed=78)
    r = RHOS[np.arange(B) % 4]
    s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
    s.set_options(FCCQPOptionsB(**LOG_OPTS))
    rho = r.copy()
    s.set_rho(rho)
    s.Solve(qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)
    sol = s.GetSolution()
    z, it, st = sol.z, sol.details.n_iter, sol.details.solve_status
    kinds = ["port"] + (["ref"] if oracle.have("ref") else [])
    for k in kinds:
        for v in RHOS:
            idx = np.flatnonzero(r == v)
            sub = qp.take(idx)
            ref = oracle.Oracle(k).solve_batch(sub, warm_mode=0, nthreads=8, **dict(LOG_OPTS, rho=float(v)))
            same = it[idx] == ref["n_iter"]
            assert rel_err(z[idx][same], ref["z"][same]).max() <= Z_TOL, (k, v)
            o, oref = sub.objective(z[idx]), sub.objective(ref["z"])
            assert (np.abs(o - oref) / np.maximum(1.0, np.abs(oref)))[same].max() <= 1e-6, (k, v)
            assert np.array_equal(st[idx][same], ref["status"][same]), (k, v)
            if k == "port":
                explain_count_mismatches(sub, it[idx], ref["n_iter"], opts=dict(LOG_OPTS, rho=float(v)), z_gpu=z[idx])
            assert (~same).mean() <= 0.005, (k, v, int((~same).sum()))
        assert (it > 0).any()


def test_adaptive_rho_carried_over_a_warm_sequence(tmp_path):
    """Humanoid, B = 512, 8 warm steps with adaptive rho every 5 iterations and the returned rho fed back, against the
    C restatement lane by lane with set_rho(last_rho) before every step."""
    import torch
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    B, T, K = 512, 8, 5
    qp = syn.make_batch(syn.HUMANOID, B, seed=79)
    opts = dict(LOG_OPTS)
    port = rho_oracle.load(tmp_path)          # the restatement, reporting the rho each solve ended with
    port.set_adaptive_rho(K)
    try:
        lanes = [port.solver(qp.n, qp.m, qp.nc, qp.lambda_c_start) for _ in range(B)]
        for o in lanes:
            o.set_options(**opts)
            o.set_warm_start(True)
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
        s.set_options(FCCQPOptionsB(adapt_rho_interval=K, **opts))
        s.set_warm_start(True)
        rho = torch.full((B,), opts["rho"], dtype=torch.float64, device="cuda:0")
        s.set_rho(rho)
        apart = np.zeros(B, bool)
        rng = np.random.default_rng(80)
        moved = 0
        dv = lambda a: torch.as_tensor(a, device="cuda:0")
        for t in range(T):
            s.Solve(dv(qp.Q), dv(qp.b), dv(qp.A_eq), dv(qp.b_eq), dv(qp.friction_coeffs), dv(qp.lb), dv(qp.ub))
            sol = s.GetSolution()
            z, it = sol.z.cpu().numpy(), sol.details.n_iter.cpu().numpy()
            r_gpu = rho.cpu().numpy()
            ref_z, ref_it, ref_rho = np.empty_like(z), np.empty_like(it), np.empty(B)
            for i, o in enumerate(lanes):
                o.Solve(qp.Q[i], qp.b[i], qp.A_eq[i], qp.b_eq[i], qp.friction_coeffs[i], qp.lb[i], qp.ub[i])
                g = o.GetSolution()
                ref_z[i], ref_it[i], ref_rho[i] = g["z"], g["n_iter"], port.last_rho()
                o.set_options(opts["max_iter"], ref_rho[i], opts["eps_fcone"], opts["eps_bound"])   # set_rho(last_rho)
            apart |= it != ref_it
            ok = ~apart
            assert apart.mean() <= 0.03, (t, int(apart.sum()))
            assert rel_err(z[ok], ref_z[ok]).max() <= 1e-6, t
            assert np.allclose(r_gpu[ok], ref_rho[ok], rtol=1e-6, atol=0), t
            moved += int((ref_rho != opts["rho"]).sum())
            qp = syn.random_walk(qp, rng)
        assert moved > 0
        print(f"humanoid warm sequence: {int(apart.sum())} of {B} lanes parted ways, {moved} lane-steps ended off rho0")
    finally:
        port.set_adaptive_rho(0)


@pytest.mark.parametrize("path", ["warp-fp64", "general", "struct-split"])
def test_adaptive_uniform_array_is_the_adaptive_call(walking_log, log512, log16k, path):
    """With adaptive rho on, the uniform-valued array runs the same CTA-kernel instance as the call without it:
    bit-identical.  (The warp kernel has an instance of its own for the array: the bar of case 1 there.)"""
    make0, qp0, qp1, kw = path_case(path, walking_log, log512, log16k)

    def make():
        s = make0()
        s.options.adapt_rho_interval = 5
        return s
    want = solve_step(make, qp0, qp1, True, **kw)
    got = solve_step(make, qp0, qp1, True, rho=np.full(qp0.batch, make().options.rho), **kw)
    if path.startswith("warp"):
        assert_close(got, want, slice(None), path)
    else:
        assert_equal(got, want, slice(None), path)
    assert (got["rho"] != make().options.rho).any()           # some lanes moved their rho, and report it


@pytest.mark.parametrize("path", ["warp-fp64", "general", "struct-split", "host"])
def test_mask_and_rho(walking_log, log512, log16k, path):
    make, qp0, qp1, kw = path_case(path, walking_log, log512, log16k)
    B = qp0.batch
    warm = scattered_mask(B, 47)
    r = lane_rhos(B, make().options.rho)
    got = solve_step(make, qp0, qp1, warm, rho=r, **kw)
    for flag in (False, True):
        for v in np.unique(r):
            want = solve_step(make, qp0, qp1, flag, rho=float(v), **kw)
            assert_close(got, want, (r == v) & (warm == flag), f"{path} warm={flag} rho {v}")


def test_graph_replays_carry_rho(walking_log):
    import torch
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    dev = torch.device("cuda:0")
    B, T = 2048, 4
    qp = walking_log.tile(B)
    names = ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub")
    static = [torch.as_tensor(getattr(qp, k), device=dev).clone() for k in names]
    opts = FCCQPOptionsB(adapt_rho_interval=5, **LOG_OPTS)

    def make(rho):
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
        s.set_options(opts)
        s.time_kernel = False
        s.zero_copy_outputs = True
        s.structure = "dense"               # fully asynchronous, capturable from the first call
        s.set_rho(rho)
        return s
    rho_g = torch.full((B,), LOG_OPTS["rho"], dtype=torch.float64, device=dev)
    rho_e = rho_g.clone()
    g_s, e_s = make(rho_g), make(rho_e)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        g_s.Solve(*static)                  # cold first step, both
        e_s.Solve(*static)
    torch.cuda.synchronize()
    g_s.set_warm_start(True)
    e_s.set_warm_start(True)
    g = torch.cuda.CUDAGraph()
    snap = [a.clone() for a in g_s.GetState()] + [rho_g.clone()]
    with torch.cuda.graph(g, stream=side):
        g_s.Solve(*static)
    for a, b_ in zip(list(g_s.GetState()) + [rho_g], snap):   # (capture ran nothing: restore to be safe)
        a.copy_(b_)
    rng = np.random.default_rng(48)
    moved = False
    for t in range(T):
        qp = syn.random_walk(qp, rng)
        for st, k in zip(static, names):
            st.copy_(torch.as_tensor(getattr(qp, k), device=dev))
        if t == 2:                          # an entry changed in place between replays takes effect
            rho_g[7] = 1e-2
            rho_e[7] = 1e-2
        g.replay()
        with torch.cuda.stream(side):
            e_s.Solve(*static)
        torch.cuda.synchronize()
        gs, es = g_s.GetSolution(), e_s.GetSolution()
        assert torch.equal(gs.z, es.z) and torch.equal(gs.details.n_iter, es.details.n_iter), t
        assert torch.equal(rho_g, rho_e), t
        for a, b_ in zip(g_s.GetState(), e_s.GetState()):
            assert torch.equal(a, b_), t
        moved |= bool((rho_g != LOG_OPTS["rho"]).any())
    assert moved


@pytest.mark.parametrize("path", ["warp-fp64", "warp-fp32", "general", "struct-split", "struct-single"])
def test_invalid_entries(walking_log, log512, log16k, path):
    make, qp0, qp1, kw = path_case(path, walking_log, log512, log16k)
    B = qp0.batch
    base = make().options.rho
    r = lane_rhos(B, base)
    bad = np.array([0, 1, 2, B // 2, B - 1])
    r_bad = r.copy()
    r_bad[bad] = [0.0, -1.0, np.nan, np.inf, -0.0]
    # a mask puts bad entries on cold and on warm lanes; its cold launches (on struct-split two-stage, rho_invalid_kernel
    # included) run before its warm ones
    for warm in (False, True, scattered_mask(B, 49)):
        got = solve_step(make, qp0, qp1, warm, rho=r_bad, **kw)
        want = solve_step(make, qp0, qp1, warm, rho=r, **kw)
        assert np.array_equal(got["status"][bad], np.full(bad.size, 2)) and not got["n_iter"][bad].any(), path
        assert got["rho"][bad].tobytes() == r_bad[bad].tobytes()
        good = np.setdiff1d(np.arange(B), bad)
        assert_equal(got, want, good, f"{path} other lanes")
    # a host array with such an entry is refused before anything runs
    s = make()
    s.set_rho(np.full(qp0.batch, base))
    s.rho_lanes[3] = 0.0
    with pytest.raises(ValueError):
        s.Solve(qp1.Q, qp1.b, qp1.A_eq, qp1.b_eq, qp1.friction_coeffs, qp1.lb, qp1.ub)


def test_schedule_from_previous_changes_only_the_order(log16k):
    qp0, qp1 = log16k
    r = lane_rhos(qp0.batch, LOG_OPTS["rho"])
    for adapt in (0, 5):
        opts = dict(LOG_OPTS, adapt_rho_interval=adapt)
        want = solve_step(solver_factory(qp0, opts, structure="probe"), qp0, qp1, True, rho=r)
        got = solve_step(solver_factory(qp0, opts, structure="probe", schedule_from_previous=True), qp0, qp1, True, rho=r)
        assert_equal(got, want, slice(None), f"LPT adapt {adapt}")
        assert np.array_equal(got["rho"], want["rho"])
