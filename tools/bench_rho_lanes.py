"""Per-lane rho in warm control loops, device-resident (FCCQPBatch.set_rho(array), fccqp_batch_solve_rho).

Each data set is a warm sequence of random-walk steps (synthetic.random_walk) after one cold solve, run in three arms:
  fixed     options.rho, adaptive rho off (the reference's iteration)
  restart   adaptive rho every 5 iterations, every step restarting at options.rho (what a warm loop got without the array)
  carried   adaptive rho every 5 iterations with a [B] rho tensor that every step reads and overwrites
The arms alternate inside every step and the whole sequence is repeated --reps times; per step: CUDA-event ms (median over
repeats), mean iterations of the QPs that iterate, share at max_iter, worst cone violation.  Then the cost of routing to the
instances that keep rho per QP: one warm step with a uniform-valued array against the same step without it (adaptive rho
off).  One JSON line per row to --out, with the card name and its power limit.

    python tools/bench_rho_lanes.py --out profiles/r03_rho_lanes.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OPTS = dict(max_iter=100, rho=5e-5, eps_fcone=1e-6, eps_bound=1e-6)   # the reference's settings for the walking log
NAMES = ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub")


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                      text=True).strip()
        name, power = [v.strip() for v in out.split(",")]
        return name, power
    except Exception as e:   # (no nvidia-smi: record why)
        import torch
        return torch.cuda.get_device_name(0), f"unknown ({type(e).__name__})"


def main():
    import torch
    from fcc_qp_b200 import synthetic as syn
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    from fcc_qp_b200.logdata import load_walking_log
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=int, default=1, help="divide every batch size by this (rehearsal)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_rho_lanes.jsonl"))
    ap.add_argument("--label", default="")
    a = ap.parse_args()
    name, power = card()
    dev = torch.device("cuda:0")
    sets = [("walking_log", lambda B: load_walking_log().tile(B), 1 << 16, 16),
            ("humanoid", lambda B: syn.make_batch(syn.HUMANOID, B, seed=5), 1 << 16, 16),
            ("multicontact", lambda B: syn.make_batch(syn.MULTICONTACT, B, seed=6), 1 << 14, 32)]
    rows = []

    def emit(row):
        row.update(gpu=name, power_limit=power, label=a.label)
        rows.append(row)
        print(json.dumps(row), flush=True)

    for data, gen, B, T in sets:
        B //= a.scale
        qp = gen(B)
        rng = np.random.default_rng(7)
        steps = [qp]
        for _ in range(T):
            steps.append(syn.random_walk(steps[-1], rng))
        # (random_walk moves b and b_eq only: the matrices are uploaded once and shared by every step)
        shared = {k: torch.as_tensor(getattr(qp, k), device=dev) for k in NAMES if k not in ("b", "b_eq")}
        dsteps = [[shared[k] if k in shared else torch.as_tensor(getattr(q, k), device=dev) for k in NAMES] for q in steps]

        def mk(adapt, array):
            s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
            s.set_options(FCCQPOptionsB(adapt_rho_interval=adapt, **OPTS))
            s.time_kernel = False
            s.zero_copy_outputs = True
            if array:
                s.set_rho(torch.full((B,), OPTS["rho"], dtype=torch.float64, device=dev))
            return s
        arms = {"fixed": (0, False), "restart": (5, False), "carried": (5, True)}
        ms = {k: np.zeros((a.reps, T)) for k in arms}
        stats = {k: [None] * T for k in arms}
        for r in range(a.reps):
            solvers = {k: mk(*v) for k, v in arms.items()}
            for k, s in solvers.items():                 # step 0: cold (untimed; structure bounds cached from here on)
                s.Solve(*dsteps[0])
                s.set_warm_start(True)
            torch.cuda.synchronize()
            for t in range(T):
                for k, s in solvers.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    s.Solve(*dsteps[t + 1])
                    e1.record()
                    torch.cuda.synchronize()
                    ms[k][r, t] = e0.elapsed_time(e1)
                    if r == 0:
                        d = s.GetSolution().details
                        it = d.n_iter.cpu().numpy()
                        rho = s.rho_lanes.cpu().numpy() if s.rho_lanes is not None else None
                        stats[k][t] = dict(mean_iter_iterating=float(it[it > 0].mean()) if (it > 0).any() else 0.0,
                                           iterating=float((it > 0).mean()), at_max_iter=float((it == OPTS["max_iter"]).mean()),
                                           worst_fcone_viol=float(d.friction_cone_viol.max().item()),
                                           rho_off_start=None if rho is None else float((rho != OPTS["rho"]).mean()))
        for k in arms:
            for t in range(T):
                emit(dict(data=data, B=B, arm=k, step=t + 1, ms_median=float(np.median(ms[k][:, t])),
                          ms_all=[round(v, 4) for v in ms[k][:, t]], **stats[k][t]))
            emit(dict(data=data, B=B, arm=k, step="total", ms_median=float(np.median(ms[k].sum(1))),
                      mean_iter_iterating=float(np.mean([s_["mean_iter_iterating"] for s_ in stats[k]])),
                      at_max_iter=float(np.mean([s_["at_max_iter"] for s_ in stats[k]])),
                      worst_fcone_viol=float(max(s_["worst_fcone_viol"] for s_ in stats[k]))))

        # routing cost: a uniform-valued array (adaptive rho off) against the same warm step without it
        if data != "multicontact":
            solvers = {"no_array": mk(0, False), "uniform_array": mk(0, True)}
            for s in solvers.values():
                s.Solve(*dsteps[0])
                s.set_warm_start(True)
                s.Solve(*dsteps[1])
            state0 = {k: tuple(x.clone() for x in s.GetState()) for k, s in solvers.items()}
            times = {k: [] for k in solvers}
            for r in range(5 * a.reps + 2):
                for k, s in solvers.items():
                    for dst, src in zip(s.GetState(), state0[k]):
                        dst.copy_(src)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    s.Solve(*dsteps[2])
                    e1.record()
                    torch.cuda.synchronize()
                    if r >= 2:
                        times[k].append(e0.elapsed_time(e1))
            same = torch.equal(solvers["no_array"].GetSolution().details.n_iter,
                               solvers["uniform_array"].GetSolution().details.n_iter)
            for k in solvers:
                emit(dict(data=data, B=B, arm=k, step="routing", ms_median=float(np.median(times[k])),
                          ms_all=[round(v, 4) for v in times[k]], same_counts=bool(same)))
        del solvers, dsteps, shared
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
