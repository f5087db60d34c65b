"""Per-lane cold or warm start (fccqp_batch_desc::warm_lanes, FCCQPBatch.set_warm_start(mask)).

1. Bit-identity with uniform calls, path by path (the shared-structure path to its own bar, see assert_lanes_close):
   from the state of one cold solve, a mixed call must return, bit for bit, what a uniform cold call returns on its cold lanes and what a uniform warm call returns on its warm lanes -- z, the
   carried duals, iteration counts, status, both residuals and both violations.  Each cell first asserts that the path it
   names ran (launch count, launch geometry, structure info): a mixed call runs the launches of a uniform cold call over
   its cold lanes and those of a uniform warm call over its warm lanes.  All-ones / all-zeros masks equal
   warm_start = 1 / 0.
2. Parity with the reference semantics over a 16-step loop that resets 5-10 % of the lanes per step: one persistent
   reference object per lane, set_warm_start(mask[i]) before every solve (C restatement, and the compiled reference when
   it is built), under the bar of test_gpu_parity.py.
3. CUDA graph: a captured mixed step replayed after the mask tensor was changed in place equals the eager call.
"""
import ctypes as C

import numpy as np
import pytest

import oracle
from conftest import LOG_OPTS
from fcc_qp_b200 import synthetic as syn
from test_gpu_parity import Z_TOL, explain_count_mismatches, rel_err

pytestmark = pytest.mark.gpu
KEYS = ("z", "mu_x", "mu_c", "n_iter", "status", "res_b", "res_f", "bviol", "fviol")
RANDOM_OPTS = dict(max_iter=200, rho=1e-3, eps_fcone=1e-7, eps_bound=1e-7)
FP32_OPTS = dict(max_iter=200, rho=1e-3, eps_fcone=1e-4, eps_bound=1e-4)


def scattered_mask(B, seed, cold=0.3, edges=(4096, 8192, 12288)):
    """~30 % cold lanes, scattered, with lane 0, lane B-1 and both sides of the given chunk boundaries cold."""
    warm = np.random.default_rng(seed).random(B) >= cold
    idx = [0, B - 1] + [i for e in edges if 0 < e < B for i in (e - 1, e)]
    warm[idx] = False
    return warm


def _np(a):
    return a.cpu().numpy().copy() if hasattr(a, "cpu") else np.array(a, copy=True)


def solve_step(make, qp0, qp1, warm, device=True, Q=None, A=None):
    """A fresh solver: a cold solve of qp0 (the carried state), then one solve of qp1 with set_warm_start(warm).  Returns
    the outputs of the second solve, its launch count and what fccqp_last_launch_info / _struct_info report."""
    import torch
    from fcc_qp_b200 import _native as nat
    s = make()
    f32 = s.precision != "fp64"

    def args(qp):
        if not device:
            return [qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub]
        dt = torch.float32 if f32 else torch.float64
        t = lambda a: torch.as_tensor(a, dtype=dt, device="cuda:0")
        return [t(qp.Q) if Q is None else Q, t(qp.b), t(qp.A_eq) if A is None else A, t(qp.b_eq), t(qp.friction_coeffs),
                t(qp.lb), t(qp.ub)]

    s.set_warm_start(False)
    s.Solve(*args(qp0))
    if isinstance(warm, np.ndarray) and device:
        warm = torch.as_tensor(warm, device="cuda:0")
    s.set_warm_start(warm)
    a1 = args(qp1)
    torch.cuda.synchronize()
    n0 = nat.lib().fccqp_kernel_launch_count()
    s.Solve(*a1)
    torch.cuda.synchronize()
    launches = nat.lib().fccqp_kernel_launch_count() - n0
    sol = s.GetSolution()
    x, mux, muc = s.GetState()
    d = sol.details
    out = dict(z=sol.z, mu_x=mux, mu_c=muc, n_iter=d.n_iter, status=d.solve_status, res_b=d.eps_bounds,
               res_f=d.eps_friction_cone, bviol=d.bounds_viol, fviol=d.friction_cone_viol)
    return {k: _np(v) for k, v in out.items()}, launches, nat.last_launch_info(), nat.last_struct_info()


def assert_lanes_equal(got, want, lanes, what):
    for k in KEYS:
        g, w = got[k][lanes], want[k][lanes]
        if g.tobytes() != w.tobytes():
            bad = np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(g, w)])
            raise AssertionError(f"{what}: {k} differs on {bad.size} of {g.shape[0]} lanes (first {bad[:5].tolist()})")


def check_mixed(make, qp0, qp1, warm, launches, device=True, check_path=None, Q=None, A=None, what=""):
    """Uniform cold, uniform warm and mixed from the same carried state; `launches` = counts of (cold, warm, mixed)."""
    runs = {}
    for mode, w in (("cold", False), ("warm", True), ("mixed", warm)):
        out, n, li, si = solve_step(make, qp0, qp1, w, device=device, Q=Q, A=A)
        if launches is not None:
            assert n == launches[mode], (what, mode, n, li, si)
        if check_path is not None:
            check_path(mode, li, si)
        runs[mode] = out
    warm = np.asarray(warm, dtype=bool)
    assert warm.any() and (~warm).any()
    assert_lanes_equal(runs["mixed"], runs["cold"], ~warm, what + " cold lanes")
    assert_lanes_equal(runs["mixed"], runs["warm"], warm, what + " warm lanes")
    # the two uniform calls really differ: the check has teeth
    assert not np.array_equal(runs["cold"]["n_iter"], runs["warm"]["n_iter"]) or \
        runs["cold"]["z"].tobytes() != runs["warm"]["z"].tobytes(), what
    it = runs["mixed"]["n_iter"]
    print(f"{what}: B={warm.size} cold lanes {int((~warm).sum())}, iterating cold {(it[~warm] > 0).mean():.3f} "
          f"warm {(it[warm] > 0).mean():.3f}")
    return runs


def solver_factory(qp, opts, structure="auto", precision="fp64", device=0, **kw):
    def make():
        from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start, precision=precision, device=device)
        s.set_options(FCCQPOptionsB(**opts))
        s.structure = structure
        for k, v in kw.items():
            setattr(s, k, v)
        return s
    return make


def dense_path(mode, li, si):
    assert not si["used"], si


@pytest.fixture(scope="module")
def log16k(walking_log):
    qp0 = walking_log.tile(16384)
    return qp0, syn.random_walk(qp0, np.random.default_rng(3))


@pytest.fixture(scope="module")
def log512(walking_log):
    qp0 = walking_log.take(np.arange(512) * 3)
    return qp0, syn.random_walk(qp0, np.random.default_rng(4))


# ---- 1. bit-identity, path by path
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_warp_kernel(precision):
    n, m, nc, lcs = 14, 5, 6, 6
    qp0 = syn.random_qps(np.random.default_rng(21), 2048, n, m, nc, lcs)
    qp1 = syn.random_walk(qp0, np.random.default_rng(22))
    opts = FP32_OPTS if precision == "fp32" else RANDOM_OPTS

    def warp(mode, li, si):
        assert li["block"] == 128 and not si["used"], (li, si)  # four warps per CTA, one QP per warp
    check_mixed(solver_factory(qp0, opts, precision=precision), qp0, qp1, scattered_mask(2048, 1),
                dict(cold=1, warm=1, mixed=2), check_path=warp, what=f"warp {precision}")


@pytest.mark.parametrize("precision", ["fp64", "fp32_data"])
def test_general_kernel(log512, precision):
    qp0, qp1 = log512
    check_mixed(solver_factory(qp0, LOG_OPTS, structure="dense", precision=precision), qp0, qp1, scattered_mask(512, 2),
                dict(cold=1, warm=1, mixed=2), check_path=dense_path, what=f"general {precision}")


def test_structure_kernel_single_launch(log512):
    qp0, qp1 = log512

    def single(mode, li, si):
        assert si["used"] and si["deferred"] == 0, si
    # probe, structure-exploiting kernel, general kernel over the (empty) hand-over list; mixed: the last two per kind
    check_mixed(solver_factory(qp0, LOG_OPTS, structure="probe"), qp0, qp1, scattered_mask(512, 3),
                dict(cold=3, warm=3, mixed=5), check_path=single, what="struct single launch")


def split_path(mode, li, si):
    assert si["used"] and si["deferred"] == 0, si


def test_structure_kernel_two_stage_split(log16k):
    """Cold: probe + first stage + resume launch + general kernel; warm: probe + single launch + general; mixed: the cold
    sequence over the cold lanes and the warm one over the warm lanes after one probe."""
    qp0, qp1 = log16k
    runs = check_mixed(solver_factory(qp0, LOG_OPTS, structure="probe"), qp0, qp1, scattered_mask(16384, 4),
                       dict(cold=4, warm=3, mixed=6), check_path=split_path, what="struct two-stage")
    assert (runs["mixed"]["n_iter"] > 0).any()


def test_structure_kernel_general_fallback(log16k):
    """Caps too small: every QP goes to the general kernel, from the first stage (cold) or the single launch (warm)."""
    qp0, qp1 = log16k

    def fallback(mode, li, si):
        assert si["used"] and si["deferred"] == 16384, si
    check_mixed(solver_factory(qp0, LOG_OPTS, structure=(8, 4, 2)), qp0, qp1, scattered_mask(16384, 5),
                dict(cold=3, warm=2, mixed=5), check_path=fallback, what="struct fallback")


def test_structure_kernel_adaptive_rho_and_relaxation(log16k):
    qp0, qp1 = log16k
    opts = dict(LOG_OPTS, adapt_rho_interval=5, relaxation=1.6)
    check_mixed(solver_factory(qp0, opts, structure="probe"), qp0, qp1, scattered_mask(16384, 6),
                dict(cold=4, warm=3, mixed=6), check_path=split_path, what="struct adaptive rho + relaxation")


def test_schedule_from_previous(log16k):
    qp0, qp1 = log16k
    check_mixed(solver_factory(qp0, LOG_OPTS, structure="probe", schedule_from_previous=True), qp0, qp1,
                scattered_mask(16384, 7), dict(cold=4, warm=3, mixed=6), check_path=split_path, what="LPT order")


def shared_set():
    import torch
    from test_gpu_shared_structure import shared_batch
    qp0 = shared_batch(syn.QUADRUPED, 16384)
    qp1 = syn.random_walk(qp0, np.random.default_rng(8))
    B = qp0.batch
    Q = torch.as_tensor(qp0.Q[:1], device="cuda:0").expand(B, qp0.n, qp0.n)
    A = torch.as_tensor(qp0.A_eq[:1], device="cuda:0").expand(B, qp0.m, qp0.n)
    return qp0, qp1, Q, A


def assert_lanes_close(got, want, lanes, what):
    """The shared-structure bar (test_gpu_shared_structure.py): that path forms the pre-solve right-hand side of the first
    QP a thread block solves while it factors, and of every later one through the cached operator -- two summation
    orders -- so which QPs open a block changes the last bits of their answers (measured: the first QP of each block
    of each launch, 2 x 592 of 16384 lanes), in uniform calls as much as in mixed ones.  Counts and status must agree on
    all but a handful of lanes, z within 1e-7 relative where they do."""
    it, itr = got["n_iter"][lanes], want["n_iter"][lanes]
    same = it == itr
    assert (~same).mean() <= 0.005, (what, int((~same).sum()))
    assert rel_err(got["z"][lanes][same], want["z"][lanes][same]).max() <= 1e-7, what
    assert np.array_equal(got["status"][lanes][same], want["status"][lanes][same]), what


def test_shared_structure_path():
    """Stride-0 Q / A_eq above 4 x resident CTAs: cold takes the pre-solve + ADMM launches, warm the ADMM one, mixed the
    cold pair over its cold lanes and the warm launch over its warm lanes."""
    qp0, qp1, Q, A = shared_set()
    warm = scattered_mask(qp0.batch, 9).astype(np.uint8)      # (a uint8 mask here, bool elsewhere)
    runs = {}
    for mode, w in (("cold", False), ("warm", True), ("mixed", warm)):
        runs[mode], n, li, si = solve_step(solver_factory(qp0, LOG_OPTS), qp0, qp1, w, Q=Q, A=A)
        assert n == dict(cold=2, warm=1, mixed=3)[mode] and not si["used"], (mode, n, si)
    warm = warm.astype(bool)
    assert_lanes_close(runs["mixed"], runs["cold"], ~warm, "shared structure cold lanes")
    assert_lanes_close(runs["mixed"], runs["warm"], warm, "shared structure warm lanes")


def test_host_path_spans_several_chunks(walking_log):
    """numpy batch of 3 x 4096 QPs: the mask is staged chunk by chunk, like the carried state."""
    qp0 = walking_log.tile(12288)
    qp1 = syn.random_walk(qp0, np.random.default_rng(10))
    runs = check_mixed(solver_factory(qp0, LOG_OPTS), qp0, qp1, scattered_mask(12288, 11), None, device=False,
                       what="host path")
    assert runs["mixed"]["n_iter"].shape == (12288,)


def test_host_path_over_two_devices(walking_log):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    qp0 = walking_log.tile(24576)
    qp1 = syn.random_walk(qp0, np.random.default_rng(12))
    check_mixed(solver_factory(qp0, LOG_OPTS, device=[0, 1]), qp0, qp1, scattered_mask(24576, 13), None,
                device=False, what="two devices")


@pytest.mark.parametrize("path", ["warp", "split", "shared", "host"])
def test_degenerate_masks_equal_uniform_calls(walking_log, log16k, path):
    """All-ones mask == warm_start = 1 and all-zeros mask == warm_start = 0, bit for bit on every lane (shared-structure
    path: to its bar, see assert_lanes_close)."""
    Q = A = None
    device = True
    if path == "warp":
        qp0 = syn.random_qps(np.random.default_rng(31), 1024, 10, 4, 6, 4)
        qp1 = syn.random_walk(qp0, np.random.default_rng(32))
        make = solver_factory(qp0, RANDOM_OPTS)
    elif path == "split":
        qp0, qp1 = log16k
        make = solver_factory(qp0, LOG_OPTS, structure="probe")
    elif path == "shared":
        qp0, qp1, Q, A = shared_set()
        make = solver_factory(qp0, LOG_OPTS)
    else:
        qp0 = walking_log.tile(8192)
        qp1 = syn.random_walk(qp0, np.random.default_rng(33))
        make = solver_factory(qp0, LOG_OPTS)
        device = False
    B = qp0.batch
    everything = np.ones(B, bool)
    for uniform, mask in ((True, np.ones(B, bool)), (False, np.zeros(B, bool))):
        got, _, _, _ = solve_step(make, qp0, qp1, mask, device=device, Q=Q, A=A)
        want, _, _, _ = solve_step(make, qp0, qp1, uniform, device=device, Q=Q, A=A)
        check = assert_lanes_close if path == "shared" else assert_lanes_equal
        check(got, want, everything, f"{path} mask all {int(uniform)}")


# ---- 2. parity with one reference object per lane over a reset loop
def oracle_solve_masked(lanes, qp, warm):
    """Lane i solved by its persistent reference object after set_warm_start(warm[i]): the cold and the warm lanes
    through the per-lane entry point of the oracle, each on its own handles."""
    B, n = qp.batch, qp.n
    out = dict(z=np.empty((B, n)), n_iter=np.empty(B, np.int32), status=np.empty(B, np.int32))
    for flag in (False, True):
        idx = np.flatnonzero(warm == flag)
        if idx.size == 0:
            continue
        sub = qp.take(idx)
        Qc, Ac = oracle.colmajor_stack(sub.Q), oracle.colmajor_stack(sub.A_eq)
        b, beq, mu, lb, ub = (np.ascontiguousarray(a, dtype=np.float64)
                              for a in (sub.b, sub.b_eq, sub.friction_coeffs, sub.lb, sub.ub))
        h = (C.c_void_p * idx.size)(*[lanes.handles[i] for i in idx])
        z = np.empty((idx.size, n)); it = np.empty(idx.size, np.int32); st = np.empty(idx.size, np.int32)
        det = np.empty((idx.size, 6))
        p, ip = oracle._ptr, oracle._ip
        lanes.o.fn("solve_lanes")(h, int(idx.size), int(flag), p(Qc), p(b), p(Ac), p(beq), p(mu), mu.shape[1], p(lb),
                                  p(ub), n, p(z), p(it, ip), p(st, ip), p(det))
        out["z"][idx], out["n_iter"][idx], out["status"][idx] = z, it, st
    return out


@pytest.mark.parametrize("data", ["walking_log", "humanoid"])
def test_reset_loop_matches_one_reference_object_per_lane(walking_log, data):
    import torch
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    B, T = 1024, 16
    qp = walking_log.take(np.arange(B)) if data == "walking_log" else syn.make_batch(syn.HUMANOID, B, seed=77)
    rng = np.random.default_rng(2024)
    kinds = ["port"] + (["ref"] if oracle.have("ref") else [])
    refs = {}
    for k in kinds:
        refs[k] = oracle.Oracle(k).lanes(B, qp.n, qp.m, qp.nc, qp.lambda_c_start)
        refs[k].set_options(**LOG_OPTS)
    s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
    s.set_options(FCCQPOptionsB(**LOG_OPTS))
    mask = torch.zeros(B, dtype=torch.bool, device="cuda:0")     # step 0: every lane cold
    s.set_warm_start(mask)
    diverged = np.zeros(B, bool)   # lanes whose count differed at an earlier step (they carry their own state since)
    n_diff = 0
    state = None
    for t in range(T):
        warm = np.zeros(B, bool) if t == 0 else rng.random(B) >= rng.uniform(0.05, 0.10)
        mask.copy_(torch.as_tensor(warm, device="cuda:0"))
        dv = lambda a: torch.as_tensor(a, device="cuda:0")
        s.Solve(dv(qp.Q), dv(qp.b), dv(qp.A_eq), dv(qp.b_eq), dv(qp.friction_coeffs), dv(qp.lb), dv(qp.ub))
        sol = s.GetSolution()
        z, it, st = sol.z.cpu().numpy(), sol.details.n_iter.cpu().numpy(), sol.details.solve_status.cpu().numpy()
        diverged &= warm                 # a cold solve ignores the carried state: the lane is in step again
        for k in kinds:
            ref = oracle_solve_masked(refs[k], qp, warm)
            same = (it == ref["n_iter"]) & ~diverged
            assert rel_err(z[same], ref["z"][same]).max() <= Z_TOL, (k, t)
            o, oref = qp.objective(z), qp.objective(ref["z"])
            assert (np.abs(o - oref) / np.maximum(1.0, np.abs(oref)))[same].max() <= 1e-6, (k, t)
            assert np.array_equal(st[same], ref["status"][same]), (k, t)
            if k == "port":
                # differing counts, and lanes that diverged earlier: the restatement from the state the GPU started from
                # (cold lanes from nothing) reproduces the GPU count and z, or the exit test sits on its threshold
                for flag in (False, True):
                    idx = np.flatnonzero(warm == flag)
                    if idx.size == 0:
                        continue
                    sub_state = None if not flag else tuple(a[idx] for a in state)
                    explain_count_mismatches(qp.take(idx), it[idx], ref["n_iter"][idx], state=sub_state, z_gpu=z[idx],
                                             also=np.flatnonzero(diverged[idx]))
                n_diff += int((it != ref["n_iter"]).sum())
                diverged |= it != ref["n_iter"]
        state = tuple(a.cpu().numpy().copy() for a in s.GetState())
        qp = syn.random_walk(qp, rng)
    print(f"{data}: {n_diff} lane-steps with a count difference of {T * B}, {int(diverged.sum())} lanes diverged at the end")
    assert n_diff <= 0.005 * T * B


# ---- 3. CUDA graph: the mask is read when the graph runs
def test_graph_replay_reads_the_mask_in_place(walking_log):
    import torch
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    dev = torch.device("cuda:0")
    B = 2048
    qp = walking_log.tile(B)
    names = ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub")
    static = [torch.as_tensor(getattr(qp, k), device=dev).clone() for k in names]
    mask = torch.zeros(B, dtype=torch.bool, device=dev)

    def make():
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
        s.set_options(FCCQPOptionsB(**LOG_OPTS))
        s.time_kernel = False
        s.zero_copy_outputs = True
        return s
    s = make()
    s.set_warm_start(mask)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        s.Solve(*static)                 # all cold: the first step, and the warm-up (structure probe, allocations)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        s.Solve(*static)
    sol = s.GetSolution()
    rng = np.random.default_rng(40)
    for r in range(3):
        qp = syn.random_walk(qp, rng)
        for t, k in zip(static, names):
            t.copy_(torch.as_tensor(getattr(qp, k), device=dev))
        warm = rng.random(B) >= 0.3
        mask.copy_(torch.as_tensor(warm, device=dev))
        before = tuple(a.clone() for a in s.GetState())
        g.replay()
        torch.cuda.synchronize()
        got = dict(z=sol.z.clone(), n_iter=sol.details.n_iter.clone(), status=sol.details.solve_status.clone(),
                   state=tuple(a.clone() for a in s.GetState()))
        e = make()
        e.structure = tuple(s._caps)       # the bounds the captured call was sized with
        e.SetState(*before)
        e.set_warm_start(mask.clone())
        e.Solve(*static)
        torch.cuda.synchronize()
        ref = e.GetSolution()
        assert torch.equal(got["z"], ref.z), r
        assert torch.equal(got["n_iter"], ref.details.n_iter) and torch.equal(got["status"], ref.details.solve_status), r
        for a, b_ in zip(got["state"], e.GetState()):
            assert torch.equal(a, b_), r
