"""Developer check of the structure-exploiting kernel against the goldens and the general kernel.
usage: python tools/struct_debug.py [B_time]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import numpy as np, torch
from fcc_qp_b200.logdata import load_walking_log
from fcc_qp_b200 import synthetic, _native as nat
from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB

G = os.path.join(ROOT, "tests", "golden")
dev = torch.device("cuda:0")
OPTS = FCCQPOptionsB(100, 5e-5, 1e-6, 1e-6)


def rel(z, zr):
    return np.abs(z - zr).max(1) / np.maximum(1.0, np.abs(zr).max(1))


def run(qp, structure, refine=False):
    s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
    s.set_options(OPTS)
    s.structure = structure
    s.refine = refine
    args = [torch.as_tensor(a, device=dev) for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
    s.Solve(*args)
    torch.cuda.synchronize()
    sol = s.GetSolution()
    info = nat.last_struct_info()
    return sol.z.cpu().numpy(), sol.details.n_iter.cpu().numpy(), sol.details.solve_status.cpu().numpy(), info, sol.details.device_time


def case(name, qp, gold):
    for refine in (True, False):
        z, it, st, info, dt = run(qp, "probe", refine)
        e = rel(z, gold["z"])
        mis = int((it != gold["n_iter"]).sum())
        print(f"{name} struct refine={int(refine)}: info={info} max_rel={e.max():.3e} p50={np.median(e):.3e} "
              f"n_iter mismatches={mis}/{len(it)} status2={(st == 2).sum()} nan={np.isnan(z).any()}", flush=True)
        if mis:
            idx = np.nonzero(it != gold["n_iter"])[0][:8]
            print("   first mismatches", [(int(i), int(it[i]), int(gold["n_iter"][i])) for i in idx])
    z, it, st, info, dt = run(qp, "dense")
    e = rel(z, gold["z"])
    print(f"{name} dense: info={info} max_rel={e.max():.3e} mismatches={(it != gold['n_iter']).sum()}", flush=True)


log = load_walking_log()
case("log", log, np.load(os.path.join(G, "walking_cold.npz")))
for shp, B in ((synthetic.HUMANOID, 192), (synthetic.QUADRUPED, 192), (synthetic.MULTICONTACT, 96)):
    case(shp.name, synthetic.make_batch(shp, B), np.load(os.path.join(G, f"synthetic_{shp.name}_cold.npz")))

# timing, device resident
Bt = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
for name, qp in (("log", log.tile(Bt)), ("humanoid", synthetic.make_batch(synthetic.HUMANOID, Bt // 4)),
                 ("quadruped", synthetic.make_batch(synthetic.QUADRUPED, Bt)),
                 ("multicontact", synthetic.make_batch(synthetic.MULTICONTACT, Bt // 4))):
    args = [torch.as_tensor(a, device=dev) for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
    for structure, refine in (("auto", True), ("auto", False), ("dense", True)):
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start); s.set_options(OPTS); s.structure = structure; s.refine = refine
        ts = []
        for r in range(4):
            s.Solve(*args); torch.cuda.synchronize()
            ts.append(s.GetSolution().details.device_time)
        t = min(ts[1:])
        print(f"time {name} B={qp.batch} {structure} refine={int(refine)}: {t*1e3:.3f} ms -> {qp.batch/t/1e6:.3f} M QP/s "
              f"launch={nat.last_launch_info()} struct={nat.last_struct_info()}", flush=True)
