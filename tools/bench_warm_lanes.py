"""Per-lane cold or warm start against its alternatives, device-resident (FCCQPBatch.set_warm_start(mask)).

From the state of one cold solve, the next step (b and b_eq after a random-walk step) is timed as: uniform cold, uniform warm,
one mixed call with 5 % and with 50 % of the lanes reset, and the workaround without a mask (gather the reset lanes, one
cold call on them and one warm call on the rest, scatter the results back).  CUDA-event time of the whole step, median of
--reps.  Also prints a digest of the uniform calls' outputs, so that two builds can be compared bit for bit.  One JSON
line per (data set, mode) to --out, with the card name and its power limit.

    python tools/bench_warm_lanes.py --out profiles/r03_warm_lanes.jsonl [--label new]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OPTS = dict(max_iter=100, rho=5e-5, eps_fcone=1e-6, eps_bound=1e-6)   # the reference's settings for the walking log


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
    from fcc_qp_b200 import _native as nat
    from fcc_qp_b200 import synthetic as syn
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
    from fcc_qp_b200.logdata import load_walking_log
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 16)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_warm_lanes.jsonl"))
    ap.add_argument("--label", default="")
    a = ap.parse_args()
    has_mask = any(f[0] == "warm_lanes" for f in nat.BatchDesc._fields_)
    name, power = card()
    dev = torch.device("cuda:0")
    B = a.batch
    sets = {"walking_log": load_walking_log().tile(B), "humanoid": syn.make_batch(syn.HUMANOID, B, seed=5)}
    rows = []
    for data, qp0 in sets.items():
        qp1 = syn.random_walk(qp0, np.random.default_rng(1))
        t = lambda x: torch.as_tensor(x, device=dev)
        in0 = [t(getattr(qp0, k)) for k in ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub")]
        in1 = [t(getattr(qp1, k)) for k in ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub")]

        def mk():
            s = FCCQPBatch(qp0.n, qp0.m, qp0.nc, qp0.lambda_c_start)
            s.set_options(FCCQPOptionsB(**OPTS))
            s.time_kernel = False
            s.zero_copy_outputs = True
            return s
        s = mk()
        s.Solve(*in0)
        s.Solve(*in0)                              # (structure bounds cached from here on)
        state0 = tuple(x.clone() for x in s.GetState())
        rng = np.random.default_rng(2)
        masks = {f: torch.as_tensor(rng.random(B) >= f, device=dev) for f in (0.05, 0.5)}
        subs = {}

        def restore(solver):
            for dst, src in zip(solver.GetState(), state0):
                dst.copy_(src)

        def uniform(warm):
            s.set_warm_start(warm)
            s.Solve(*in1)

        def mixed(f):
            s.set_warm_start(masks[f])
            s.Solve(*in1)

        def workaround(f):
            # without a mask: gather the reset lanes and the others, one cold and one warm call, scatter back
            w = masks[f]
            ic, iw = torch.nonzero(~w).squeeze(1), torch.nonzero(w).squeeze(1)
            if f not in subs:
                subs[f] = (mk(), mk())
            sc, sw = subs[f]
            x, mux, muc = state0
            sw.SetState(x.index_select(0, iw), mux.index_select(0, iw), muc.index_select(0, iw))
            sc.set_warm_start(False)
            sc.Solve(*[v.index_select(0, ic) for v in in1])
            sw.set_warm_start(True)
            sw.Solve(*[v.index_select(0, iw) for v in in1])
            for full, c_, w_ in zip(s.GetState(), sc.GetState(), sw.GetState()):
                full.index_copy_(0, ic, c_)
                full.index_copy_(0, iw, w_)
            for k in ("n_iter", "solve_status", "eps_bounds", "eps_friction_cone", "bounds_viol", "friction_cone_viol"):
                full = getattr(s.GetSolution().details, k)
                full.index_copy_(0, ic, getattr(sc.GetSolution().details, k))
                full.index_copy_(0, iw, getattr(sw.GetSolution().details, k))

        modes = {"cold": lambda: uniform(False), "warm": lambda: uniform(True)}
        if has_mask:
            modes.update({"mixed_5pct": lambda: mixed(0.05), "mixed_50pct": lambda: mixed(0.5)})
        modes.update({"workaround_5pct": lambda: workaround(0.05), "workaround_50pct": lambda: workaround(0.5)})
        for mode, fn in modes.items():
            times = []
            for r in range(a.reps + 2):                # two untimed: allocations, structure probes of the subsets
                restore(s)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                if r >= 2:
                    times.append(e0.elapsed_time(e1))
            sol = s.GetSolution()
            x, mux, muc = s.GetState()
            digest = hashlib.sha256()
            for v in (sol.z, sol.details.n_iter, sol.details.solve_status, mux, muc, sol.details.eps_bounds):
                digest.update(v.cpu().numpy().tobytes())
            it = sol.details.n_iter.cpu().numpy()
            row = dict(data=data, mode=mode, B=B, ms_median=float(np.median(times)), ms_min=float(np.min(times)),
                       ms_all=[round(v, 4) for v in times], mqps=B / float(np.median(times)) / 1e3,
                       iterating=float((it > 0).mean()), mean_iter=float(it.mean()), digest=digest.hexdigest()[:16],
                       gpu=name, power_limit=power, label=a.label)
            rows.append(row)
            print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
