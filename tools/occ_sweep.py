"""Occupancy sweep: M QP/s of the tiled walking log against resident CTAs per SM (FCCQP_CTAS_PER_SM is read once per
process, so one subprocess per point).  usage: python tools/occ_sweep.py [B]"""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = sys.argv[1] if len(sys.argv) > 1 else "32768"
code = r'''
import os, sys; sys.path.insert(0, sys.argv[1])
import torch
from fcc_qp_b200.logdata import load_walking_log
from fcc_qp_b200 import synthetic
from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
from fcc_qp_b200 import _native as nat
B = int(sys.argv[2]); shape = sys.argv[3]; structure = sys.argv[4]
qp = load_walking_log().tile(B) if shape == "log" else synthetic.make_batch(synthetic.SHAPES[shape], B)
args = [torch.as_tensor(a, device="cuda:0") for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start); s.set_options(FCCQPOptionsB(100, 5e-5, 1e-6, 1e-6)); s.structure = structure
ts = []
for r in range(4):
    s.Solve(*args); torch.cuda.synchronize(); ts.append(s.GetSolution().details.device_time)
t = min(ts[1:]); li = nat.last_launch_info()
print(f"{shape} {structure} ctas/SM={li['ctas_per_sm']} threads={li['block']}: {t*1e3:.3f} ms {B/t/1e6:.3f} M QP/s  per-QP latency {li['grid']*t/B*1e6:.1f} us", flush=True)
'''
for shape, structure in (("log", "auto"), ("log", "dense"), ("quadruped", "auto")):
    for c in (1, 2, 3, 4, 5, 6, 8):
        env = dict(os.environ, FCCQP_CTAS_PER_SM=str(c))
        subprocess.run([sys.executable, "-c", code, ROOT, B, shape, structure], env=env)
