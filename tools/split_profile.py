"""Per-kernel device time of the two-stage cold solve of the tiled walking log (torch.profiler, CUDA activities):
the structure probe, the first-stage kernel, the resume kernel and the general kernel, and how many QPs the first
stage left to the resume kernel.
usage: python tools/split_profile.py [B] [reps] [out.json]"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

from fcc_qp_b200 import _native as nat
from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
from fcc_qp_b200.logdata import load_walking_log

B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
out = sys.argv[3] if len(sys.argv) > 3 else None

qp = load_walking_log().tile(B)
dev = torch.device("cuda:0")
args = [torch.as_tensor(a, device=dev) for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
s.set_options(FCCQPOptionsB(100, 5e-5, 1e-6, 1e-6))
s.time_kernel = False
for _ in range(3):
    s.Solve(*args)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(reps):
        s.Solve(*args)
    torch.cuda.synchronize()
it = s.GetSolution().details.n_iter.cpu().numpy()
info = nat.last_struct_info()


def stage(name):
    if "fccqp_struct_probe_kernel" in name:
        return "probe"
    if "fccqp_struct_kernel" in name:
        # template arguments <threads, min blocks, adapt, stage>: 1 and 2 first stage; 0 the full kernel (the resume
        # launch of a two-stage solve, or the single launch)
        stage = name.replace(" ", "").split("(")[0].rstrip(">").split(",")[-1]
        return "first stage" if stage in ("1", "2") else "full / resume"
    if "fccqp_solve_kernel" in name:
        return "general"
    return None


rows = {}
for e in prof.key_averages():
    st = stage(e.key)
    if st is None:
        continue
    t = getattr(e, "device_time_total", None)
    if t is None:
        t = e.cuda_time_total
    r = rows.setdefault(st, dict(kernel=e.key, calls=0, us_total=0.0))
    r["calls"] += e.count
    r["us_total"] += t
for r in rows.values():
    r["ms_per_solve"] = r["us_total"] / reps / 1e3
res = dict(B=B, reps=reps, device=torch.cuda.get_device_name(0), kernels=rows,
           resumed=int((it > 0).sum()), ran_all_iterations=int((it == 100).sum()), deferred=info["deferred"],
           mean_iters=float(it.mean()))
print(json.dumps(res, indent=1))
if out:
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
