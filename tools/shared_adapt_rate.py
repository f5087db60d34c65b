"""Cost of adaptive rho on a shared-structure batch (one Q and one A_eq, batch stride 0).  The cached-factorization path
has no adaptive instance, so a stride-0 batch with adapt_rho_interval > 0 runs on the structure-exploiting kernel.  Rates
of a multi-contact batch for: K = 5 at stride 0, K = 0 at stride 0 (shared path), K = 5 on the materialised batch.
usage: python tools/shared_adapt_rate.py [B]   (2048 command draws around one linearisation, tiled to B; default 2^16)"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
from fcc_qp_b200 import synthetic as syn
from fcc_qp_b200 import _native as nat
from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB
from test_gpu_shared_structure import shared_batch

B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
dev = torch.device("cuda:0")
qp = shared_batch(syn.MULTICONTACT, 2048).tile(B)
vec = [torch.as_tensor(a, device=dev) for a in (qp.b, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
Q1, A1 = torch.as_tensor(qp.Q[0], device=dev), torch.as_tensor(qp.A_eq[0], device=dev)
stride0 = (Q1.expand(B, qp.n, qp.n), A1.expand(B, qp.m, qp.n))
full = (Q1.expand(B, qp.n, qp.n).contiguous(), A1.expand(B, qp.m, qp.n).contiguous())
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
for label, K, (Q, A) in (("stride0_K5", 5, stride0), ("stride0_K0_shared", 0, stride0), ("materialised_K5", 5, full)):
    s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start)
    s.set_options(FCCQPOptionsB(100, 5e-5, 1e-6, 1e-6, 1.0, K))
    times = []
    for i in range(8):
        n0 = nat.lib().fccqp_kernel_launch_count()
        ev[0].record()
        s.Solve(Q, vec[0], A, vec[1], vec[2], vec[3], vec[4])
        ev[1].record()
        torch.cuda.synchronize()
        if i >= 2:                           # the first calls load modules and probe the structure
            times.append(ev[0].elapsed_time(ev[1]) * 1e-3)
    it = s.GetSolution().details.n_iter.cpu().numpy()
    t = float(np.median(times))
    print(json.dumps({"case": label, "batch": B, "adapt_rho_interval": K, "gpu": gpu, "median_ms": 1e3 * t,
                      "M_qps_per_s": B / t / 1e6, "launches": nat.lib().fccqp_kernel_launch_count() - n0,
                      "struct_used": nat.last_struct_info()["used"], "max_iter_fraction": float((it == 100).mean())}),
          flush=True)
