"""Two-stage cold solves of the structure-exploiting kernel (fcc_qp_b200/csrc/fccqp_struct.cuh, launch_struct): a cold
batch of at least 8 QPs per resident CTA runs a first-stage kernel through the exit test of iteration 0 and
has the full kernel resume the QPs that keep iterating.  Every QP goes through the same arithmetic in the same order
as in the single launch that smaller batches take, so every output must be bit-identical to solving the same QPs in
batches below the threshold."""
import numpy as np
import pytest

from conftest import LOG_OPTS

pytestmark = pytest.mark.gpu

CHUNK = 128   # below the resident CTAs of any instance on a B200: single launch


def _solve(qp, lo, hi, opts, structure, refine, layout, lpt):
    import torch
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
    s.set_options(FCCQPOptionsB(**opts))
    s.structure = structure
    s.refine = refine
    s.schedule_from_previous = lpt
    args = [layout(torch.as_tensor(a[lo:hi], device="cuda:0")) if a.ndim == 3 else
            torch.as_tensor(a[lo:hi], device="cuda:0")
            for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
    for _ in range(2 if lpt else 1):   # LPT orders the second solve by the iteration counts of the first
        s.Solve(*args)
    torch.cuda.synchronize()
    sol = s.GetSolution()
    x, mux, muc = s.GetState()
    d = sol.details
    out = dict(z=sol.z, n_iter=d.n_iter, status=d.solve_status, res_b=d.eps_bounds, res_f=d.eps_friction_cone,
               bviol=d.bounds_viol, fviol=d.friction_cone_viol, x=x, mu_x=mux, mu_c=muc)
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def row_major(t):
    return t.contiguous()


def column_major(t):
    return t.transpose(1, 2).contiguous().transpose(1, 2)


def strided(t):
    import torch
    big = torch.zeros(t.shape[0], t.shape[1], t.shape[2] + 3, dtype=t.dtype, device=t.device)
    big[:, :, : t.shape[2]] = t
    return big[:, :, : t.shape[2]]


def check_split(qp, opts=LOG_OPTS, structure="probe", refine=False, layout=row_major, lpt=False, launches=4):
    from fcc_qp_b200 import _native as nat
    B = qp.batch
    n0 = nat.lib().fccqp_kernel_launch_count()
    big = _solve(qp, 0, B, opts, structure, refine, layout, lpt)
    assert nat.lib().fccqp_kernel_launch_count() - n0 == launches * (2 if lpt else 1)
    info = nat.last_struct_info()
    # the chunks use the bounds the large batch was solved with: both take the same QPs to the general kernel
    caps = tuple(info["caps"]) if info["used"] else structure
    parts = [_solve(qp, lo, min(lo + CHUNK, B), opts, caps, refine, layout, lpt) for lo in range(0, B, CHUNK)]
    for k, v in big.items():
        ref = np.concatenate([p[k] for p in parts])
        assert v.tobytes() == ref.tobytes(), f"{k} differs between the two-stage and the single-launch solve"
    return big, info


@pytest.fixture(scope="module")
def log8k(walking_log):
    return walking_log.tile(8192)


def test_split_walking_log(log8k):
    out, info = check_split(log8k)
    assert info["used"] and info["deferred"] == 0
    assert (out["n_iter"] > 0).any()          # some QPs went through the resume launch


@pytest.mark.parametrize("max_iter", [0, 1, 2])
def test_split_max_iter(log8k, max_iter):
    check_split(log8k, opts=dict(LOG_OPTS, max_iter=max_iter))


def test_split_relaxation(log8k):
    check_split(log8k, opts=dict(LOG_OPTS, relaxation=1.6))


def test_split_adaptive_rho_every_iteration(log8k):
    check_split(log8k, opts=dict(LOG_OPTS, adapt_rho_interval=1))


def test_split_refine(log8k):
    check_split(log8k, refine=True)


@pytest.mark.parametrize("layout", [column_major, strided])
def test_split_layouts(log8k, layout):
    check_split(log8k, layout=layout)


def test_split_lpt_order(log8k):
    check_split(log8k, lpt=True)


def test_split_caps_too_small(walking_log):
    """Caps below the log's structure: the first stage hands every QP to the general kernel.  (These caps select the
    64-thread instance, which holds more CTAs per SM: a larger batch is needed to split.)"""
    qp = walking_log.tile(16384)
    _, info = check_split(qp, structure=(8, 4, 2), launches=3)
    assert info["deferred"] == qp.batch


def test_split_unstructured_qps_go_to_the_general_kernel(log8k):
    qp = log8k.take(np.arange(log8k.batch))
    dense = np.arange(5, qp.batch, 37)
    qp.Q[dense] += 1e-3   # rank-one PSD coupling: no variable is separable any more
    _, info = check_split(qp, structure=(23, 11, 6), launches=3)
    assert info["deferred"] >= len(dense)


@pytest.mark.parametrize("shape", ["humanoid", "multicontact"])
def test_split_synthetic_sets(shape):
    from fcc_qp_b200.synthetic import SHAPES, make_batch
    qp = make_batch(SHAPES[shape], 8192, seed=7)
    out, info = check_split(qp)
    assert info["used"]
    assert (out["n_iter"] > 0).mean() > 0.05
