#!/usr/bin/env python
"""Headline benchmark: QPs solved per second at batch 2^16 per GPU (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

`--dump-outputs DIR` writes what the last timed step returned (rank 0's shard) as DIR/<name>.npy, float64:
the inputs depend on the arguments only, so two builds can be compared output for output.

One "step" = one cold batched Solve of 65 536 QPs per GPU: the 2019 logged Cassie walking QPs
(tests/golden/walking_log_compact.npz) tiled to 2^16 (SURVEY.md 8d config 2), solver settings of
fcc_qp_test.py:78-83 (rho 5e-5, eps 1e-6, max_iter 100).  Weak scaling: every rank owns its own
2^16 QPs, no data-path collective (SURVEY.md 8e).

`value`  : whole-job QP/s with inputs resident in HBM, CUDA events on the launching stream.
`e2e`    : the same through the public API (FCCQPBatch.Solve on pinned HOST arrays -> C ABI),
           host->device and device->host copies inside the timed region.
`--impl reference` times the reference's own CPU implementation (oracle/_ref: the unmodified
reference compiled from /root/reference; else the C restatement) on all host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from fcc_qp_b200 import sharding  # noqa: E402
from fcc_qp_b200.logdata import load_walking_log  # noqa: E402

BATCH_PER_GPU = 1 << 16
OPTS = dict(max_iter=100, rho=5e-5, eps_fcone=1e-6, eps_bound=1e-6)  # fcc_qp_test.py:78-83
METRIC = "qps_solved_per_sec_batch_65536_cold"
WORKLOAD = "walking_log_tiled_to_2^16_per_gpu_cold_fp64"


def algorithmic_bytes_per_qp(n, m, nc):
    """SURVEY.md 8d: FP64 bytes in = 8(n^2 + mn + 3n + m + nc/3), out = 8n + 40."""
    return 8 * (n * n + m * n + 3 * n + m + nc // 3) + 8 * n + 40


def algorithmic_flops_per_qp(n, m, iters_executed, cold=True):
    """SURVEY.md 8d: (1/3)N^3 per factorization (x2 cold) + 2N^2 per executed iteration."""
    N = n + m
    return (2 if cold else 1) * N ** 3 / 3.0 + 2.0 * N * N * iters_executed


def dump_outputs(path, sol):
    """The arrays FCCQPBatch.GetSolution() returned, one float64 .npy each (n_iter and solve_status are exact
    in float64): about 35 MB at 2^16 QPs of the walking log."""
    os.makedirs(path, exist_ok=True)
    d = sol.details
    arrays = {"z": sol.z, "n_iter": d.n_iter, "solve_status": d.solve_status, "eps_bounds": d.eps_bounds,
              "eps_friction_cone": d.eps_friction_cone, "bounds_viol": d.bounds_viol,
              "friction_cone_viol": d.friction_cone_viol}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy().astype(np.float64))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"  # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nme, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(qp, sample, nthreads=None, kind=None, warm_mode=0):
    """All-core CPU solve of the first `sample` QPs (cold, or warm-sequential inside each thread's chunk);
    returns (qps_per_s, cores, kind, seconds).  kind: "reference" (oracle/_ref, the reference's own flags),
    "reference_avx2" (same sources, -march=x86-64-v3) or "port" (the C restatement)."""
    from oracle import Oracle, colmajor_stack, have
    if kind is None:
        kind = "reference" if have("ref") else "port"
    orc = Oracle({"reference": "ref", "reference_avx2": "ref_avx2", "port": "port"}[kind])
    cores = nthreads or orc.hardware_threads()
    sub = qp.take(np.arange(sample) % qp.batch)
    prepared = (colmajor_stack(sub.Q), colmajor_stack(sub.A_eq))  # layout prep outside the timed region
    r = orc.solve_batch(sub, warm_mode=warm_mode, nthreads=cores, prepared=prepared, **OPTS)
    return sample / r["elapsed"], cores, kind, r["elapsed"]


def cpu_baseline_variants(log, sample):
    """BASELINE.md section 3 extras, reported next to (never instead of) the cold reference-flags baseline: the
    reference in its deployment mode (warm-started inside each thread's chunk of consecutive log QPs) and a second
    build with the host's vector ISA enabled.  The AVX2 build runs in a child process: an illegal instruction on
    an older host must not take the bench down."""
    from oracle import have
    out = {}
    try:
        rate, cores, kind, secs = cpu_reference_run(log, sample, warm_mode=1)
        out["warm_within_chunk"] = {"value": rate, "unit": "QP/s", "cores": cores, "kind": kind,
                                    "sample": f"first {sample} QPs, each thread warm-starts through its chunk, {secs:.1f} s"}
    except Exception as e:  # pragma: no cover
        out["warm_within_chunk"] = {"unavailable": repr(e)}
    if have("ref_avx2"):
        code = ("import sys, json; sys.path.insert(0, %r); import bench; from fcc_qp_b200.logdata import load_walking_log; "
                "log = load_walking_log(); r = {}; "
                "[r.__setitem__(k, bench.cpu_reference_run(log, %d, kind='reference_avx2', warm_mode=w)[:2]) for k, w in (('cold', 0), ('warm', 1))]; "
                "print('RESULT ' + json.dumps(r))" % (ROOT, sample))
        try:
            cp = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=180)
            res = [l for l in cp.stdout.splitlines() if l.startswith("RESULT ")]
            if cp.returncode == 0 and res:
                r = json.loads(res[-1][7:])
                out["reference_avx2"] = {"cold": {"value": r["cold"][0], "unit": "QP/s", "cores": r["cold"][1]},
                                         "warm_within_chunk": {"value": r["warm"][0], "unit": "QP/s", "cores": r["warm"][1]},
                                         "flags": "-O3 -DNDEBUG -march=x86-64-v3", "sample": f"first {sample} QPs"}
            else:
                out["reference_avx2"] = {"unavailable": f"child exited {cp.returncode}: {cp.stderr.strip()[-200:]}"}
        except Exception as e:  # pragma: no cover
            out["reference_avx2"] = {"unavailable": repr(e)}
    else:
        out["reference_avx2"] = {"unavailable": "oracle/_ref/libfccqp_ref_avx2.so not built"}
    return out


def shape_extras(dev):
    """BASELINE.json configs 3-5 on this GPU, device-resident (extra keys; the headline stays config 2).
    Synthetic QPs of the named shapes (fcc_qp_b200/synthetic.py): 4096 distinct ones generated on the host and tiled
    on the device to the batch the config states."""
    import torch
    from fcc_qp_b200 import synthetic as syn
    from fcc_qp_b200 import _native as nat
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB

    def device_batch(qp, B):
        reps = B // qp.batch
        t = [torch.as_tensor(a, device=dev) for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
        return [a.repeat((reps,) + (1,) * (a.dim() - 1)) for a in t]

    def rate(s, args, B, warm):
        best = 1e9
        for _ in range(3):
            if warm:      # warm solve of the same problems from the converged state of a cold solve
                s.set_warm_start(False); s.Solve(*args); s.set_warm_start(True)
            s.Solve(*args); torch.cuda.synchronize(dev)
            best = min(best, s.GetSolution().details.device_time)
        it = s.GetSolution().details.n_iter.cpu().numpy()
        return {"ms": 1e3 * best, "qps": B / best, "iterating_fraction": float((it > 0).mean()),
                "max_iter_fraction": float((it == OPTS["max_iter"]).mean()), "mean_iterations": float(it.mean())}

    out = {}
    for name, B, cfg in (("humanoid", 1 << 16, 3), ("quadruped", 1 << 17, 4)):
        try:
            qp = syn.make_batch(syn.SHAPES[name], 4096)
            args = device_batch(qp, B)
            s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start, device=dev.index); s.set_options(FCCQPOptionsB(**OPTS))
            s.set_warm_start(False); s.Solve(*args); torch.cuda.synchronize(dev)
            out[name] = {"baseline_config": cfg, "n": qp.n, "m": qp.m, "nc": qp.nc, "batch": B,
                         "cold": rate(s, args, B, False), "warm": rate(s, args, B, True),
                         "launch": nat.last_launch_info(), "structure": nat.last_struct_info()}
            if cfg == 4:
                out[name]["note"] = "config 4 is 2^20 QPs over 8 GPUs: this is one GPU's 2^17 share"
            del args, s
        except Exception as e:  # pragma: no cover
            out[name] = {"error": repr(e)}
    # small QPs: the warp-per-QP kernel (n + m <= 32; fccqp_warp.cuh), random well-conditioned QPs at the settings of
    # fccqp.pdf Table 1 (max_iter 15, eps 1e-4); the generator is the parity tests' own
    try:
        from fcc_qp_b200.synthetic import random_qps
        small = {}
        for (sn, sm, snc, slcs) in ((12, 6, 6, 3), (24, 8, 6, 0)):
            base = random_qps(np.random.default_rng(sn), 4096, sn, sm, snc, slcs)
            B = 1 << 18
            args = device_batch(base, B)
            s = FCCQPBatch(sn, sm, snc, slcs, device=dev.index)
            s.set_options(FCCQPOptionsB(max_iter=15, rho=1e-3, eps_fcone=1e-4, eps_bound=1e-4))
            best = 1e9
            for _ in range(3):
                s.Solve(*args); torch.cuda.synchronize(dev)
                best = min(best, s.GetSolution().details.device_time)
            it = s.GetSolution().details.n_iter.cpu().numpy()
            small[f"n{sn}_m{sm}"] = {"n": sn, "m": sm, "nc": snc, "batch": B, "ms": 1e3 * best, "qps": B / best,
                                     "mean_iterations": float(it.mean()), "launch": nat.last_launch_info()}
            # FCCQP_PRECISION_FP32: float32 data + FP32 arithmetic (stated bound in include/fccqp.h), same QPs
            z64 = s.GetSolution().z[:4096].cpu().numpy()
            args32 = [a.to(torch.float32) for a in args]
            del args, s
            s = FCCQPBatch(sn, sm, snc, slcs, device=dev.index, precision="fp32")
            s.set_options(FCCQPOptionsB(max_iter=15, rho=1e-3, eps_fcone=1e-4, eps_bound=1e-4))
            best = 1e9
            for _ in range(3):
                s.Solve(*args32); torch.cuda.synchronize(dev)
                best = min(best, s.GetSolution().details.device_time)
            z32 = s.GetSolution().z[:4096].cpu().numpy()
            err = np.abs(z32 - z64).max(axis=1) / np.maximum(1.0, np.abs(z64).max(axis=1))
            small[f"n{sn}_m{sm}"]["fp32_arithmetic"] = {"ms": 1e3 * best, "qps": B / best, "z_rel_err_max_vs_fp64": float(err.max()),
                                                        "launch": nat.last_launch_info()}
            del args32, s
        out["small_qps_warp_kernel"] = small
    except Exception as e:  # pragma: no cover
        out["small_qps_warp_kernel"] = {"error": repr(e)}
    # opt-in adaptive rho (fccqp_options::adapt_rho_interval = 5; NOT the reference's iteration) on the headline workload
    try:
        log = load_walking_log()
        qp = log.take(np.arange(1 << 16) % log.batch)
        args = [torch.as_tensor(a, device=dev) for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start, device=dev.index)
        s.set_options(FCCQPOptionsB(adapt_rho_interval=5, **OPTS))
        best = 1e9
        for _ in range(3):
            s.Solve(*args); torch.cuda.synchronize(dev)
            best = min(best, s.GetSolution().details.device_time)
        it = s.GetSolution().details.n_iter.cpu().numpy()
        out["walking_log_adaptive_rho_5"] = {"batch": 1 << 16, "ms": 1e3 * best, "qps": (1 << 16) / best,
                                             "max_iter_fraction": float((it == OPTS["max_iter"]).mean()),
                                             "mean_iterations_of_iterating": float(it[it > 0].mean()),
                                             "note": "extension, changes the iterates: not comparable with the reference's counts"}
        del args, s, qp
    except Exception as e:  # pragma: no cover
        out["walking_log_adaptive_rho_5"] = {"error": repr(e)}
    # FCCQP_SCHEDULE_LPT (FCCQPBatch.schedule_from_previous): the same cold batch solved again into the same arrays, lanes that
    # ran long in the previous solve pulled from the work queue first.  Same results bit for bit (tests); an extra key
    # because the headline `value` must not depend on a previous solve of the same data.
    try:
        log = load_walking_log()
        qp = log.take(np.arange(1 << 16) % log.batch)
        args = [torch.as_tensor(a, device=dev) for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start, device=dev.index); s.set_options(FCCQPOptionsB(**OPTS))
        s.schedule_from_previous = True
        s.Solve(*args); torch.cuda.synchronize(dev)          # no hint yet
        best = 1e9
        for _ in range(3):
            s.Solve(*args); torch.cuda.synchronize(dev)
            best = min(best, s.GetSolution().details.device_time)
        out["walking_log_schedule_from_previous"] = {"batch": 1 << 16, "ms": 1e3 * best, "qps": (1 << 16) / best,
                                                     "note": "processing order from the previous solve's iteration counts"}
        del args, s, qp
    except Exception as e:  # pragma: no cover
        out["walking_log_schedule_from_previous"] = {"error": repr(e)}
    # opt-in solution polish (FCCQPBatch.Polish: active-set guess + one more batched KKT solve + acceptance tests) on the headline
    # workload: time of the polish step next to the solve, accepted fraction, friction-cone violation of the QPs that ended at
    # max_iter before / after
    try:
        log = load_walking_log()
        qp = log.take(np.arange(1 << 16) % log.batch)
        args = [torch.as_tensor(a, device=dev) for a in (qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub)]
        s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start, device=dev.index); s.set_options(FCCQPOptionsB(**OPTS))
        s.Solve(*args); s.Polish(); torch.cuda.synchronize(dev)            # warm-up (allocations, structure probe of the inner solver)
        best = 1e9
        for _ in range(3):
            s.Solve(*args); torch.cuda.synchronize(dev)
            a = s.GetSolution()
            fv0, st0 = a.details.friction_cone_viol.clone(), a.details.solve_status.clone()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); pz = s.Polish(); e1.record(); torch.cuda.synchronize(dev)
            best = min(best, e0.elapsed_time(e1) * 1e-3)
        flag = pz.details.polished.bool()
        late = flag & (st0 == 1)
        out["walking_log_polish"] = {"batch": 1 << 16, "polish_ms": 1e3 * best, "accepted_fraction": float(flag.double().mean()),
                                     "at_max_iter": int((st0 == 1).sum()), "at_max_iter_accepted": int(late.sum()),
                                     "fcone_viol_max_before": float(fv0[late].max()) if bool(late.any()) else None,
                                     "fcone_viol_max_after": float(pz.details.friction_cone_viol[late].max()) if bool(late.any()) else None,
                                     "note": "extension (the reference has no polish step): not part of value / e2e"}
        del args, s, qp
    except Exception as e:  # pragma: no cover
        out["walking_log_polish"] = {"error": repr(e)}
    # config 5: multi-contact humanoid, T = 32 sequential warm-started batches of 2^14 (b, b_eq drift 2 % per step)
    try:
        shp = syn.SHAPES["multicontact"]
        B, T = 1 << 14, 32
        qp = syn.make_batch(shp, 2048, seed=shp.seed + 1)
        Q, b0, A, beq0, mu, lb, ub = device_batch(qp, B)

        def sequence(hint):
            s = FCCQPBatch(qp.n, qp.m, qp.nc, qp.lambda_c_start, device=dev.index); s.set_options(FCCQPOptionsB(**OPTS))
            s.schedule_from_previous = hint
            b, beq = b0, beq0
            s.Solve(Q, b, A, beq, mu, lb, ub); torch.cuda.synchronize(dev)     # untimed warm-up launch
            gen = torch.Generator(device=dev); gen.manual_seed(3)
            per = []
            for t in range(T):
                s.set_warm_start(t > 0)
                s.Solve(Q, b, A, beq, mu, lb, ub); torch.cuda.synchronize(dev)
                per.append(s.GetSolution().details.device_time)
                b = b * (1.0 + 0.02 * torch.randn(b.shape, device=dev, dtype=torch.float64, generator=gen))
                beq = beq * (1.0 + 0.02 * torch.randn(beq.shape, device=dev, dtype=torch.float64, generator=gen))
            return per, s.GetSolution().details.n_iter.cpu().numpy()

        per, it = sequence(False)
        out["multicontact"] = {"baseline_config": 5, "n": qp.n, "m": qp.m, "nc": qp.nc, "batch": B, "steps": T,
                               "total_ms": 1e3 * sum(per), "qps": B * T / sum(per), "first_cold_ms": 1e3 * per[0],
                               "cold_qps": B / per[0], "warm_ms_median": 1e3 * float(np.median(per[1:])),
                               "iterating_fraction_last": float((it > 0).mean()),
                               "launch": nat.last_launch_info(), "structure": nat.last_struct_info()}
        per, _ = sequence(True)    # FCCQP_SCHEDULE_LPT: each step's processing order from the step before
        out["multicontact"]["schedule_from_previous"] = {"total_ms": 1e3 * sum(per), "qps": B * T / sum(per),
                                                         "warm_ms_median": 1e3 * float(np.median(per[1:]))}
    except Exception as e:  # pragma: no cover
        out["multicontact"] = {"error": repr(e)}
    return out


def run_reference_arm(args):
    rank, _, world = sharding.env_rank_world()
    if rank != 0:
        return 0
    qp = load_walking_log()
    # calibrate, then size each step to a few seconds of all-core CPU work
    rate, cores, kind, _ = cpu_reference_run(qp, 2019)
    sample = int(min(BATCH_PER_GPU, max(2019, rate * 3.0)))
    for _ in range(args.warmup):
        cpu_reference_run(qp, min(sample, 4038))
    t_tot, n_tot = 0.0, 0
    for _ in range(args.steps):
        r, cores, kind, secs = cpu_reference_run(qp, sample)
        t_tot += secs; n_tot += sample
    value = n_tot / t_tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "QP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "reference walking log (2019 logged Cassie QPs) tiled",
        "config": {"workload": WORKLOAD, "sample_qps_per_step": sample, "solver": OPTS,
                   "note": "CPU reference, one FCCQP object per thread, cold solves"},
        "cpu_baseline": {"value": value, "unit": "QP/s", "cores": cores, "kind": kind,
                         "sample": f"first {sample} QPs of the tiled log per step, cold, all host threads"},
        "e2e": {"value": value, "unit": "QP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def run_ours(args):
    import torch
    from fcc_qp_b200 import _native as nat
    from fcc_qp_b200.batch import FCCQPBatch, FCCQPOptionsB

    rank, local_rank, world = sharding.init_process_group()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the solver has no CPU path (use --impl reference)")
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    log = load_walking_log()
    n, m, nc, lcs = log.n, log.m, log.nc, log.lambda_c_start
    B = BATCH_PER_GPU
    # every rank tiles the log from a different offset so that shards are not byte-identical
    idx = (np.arange(B) + rank * 997) % log.batch
    qp = log.take(idx)
    host = [qp.Q, qp.b, qp.A_eq, qp.b_eq, qp.friction_coeffs, qp.lb, qp.ub]
    dev_args = [torch.as_tensor(a, device=dev) for a in host]
    in_bytes = sum(a.nbytes for a in host)

    solver = FCCQPBatch(n, m, nc, lcs, device=local_rank)
    solver.set_options(FCCQPOptionsB(**OPTS))
    solver.time_kernel = False
    stream = torch.cuda.current_stream(dev)

    # ---------------- device-resident throughput (`value`) ----------------
    for _ in range(max(args.warmup, 3)):
        solver.Solve(*dev_args)
    torch.cuda.synchronize(dev)
    sharding.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = nat.lib().fccqp_kernel_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    torch.cuda.synchronize(dev)
    ev[0].record(stream)
    for k in range(args.steps):
        solver.Solve(*dev_args)          # asynchronous launch on the current torch stream
        ev[k + 1].record(stream)
    torch.cuda.synchronize(dev)
    sol = solver.GetSolution()           # of the last timed step (the untimed launches below replace it)
    sharding.barrier()
    launches = nat.lib().fccqp_kernel_launch_count() - launches0
    step_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    total_s = sharding.max_over_ranks(ev[0].elapsed_time(ev[-1]) * 1e-3, dev)
    # the K-step region is ~65 ms: too short for nvidia-smi's sampling period, so keep the GPU under
    # the same load until the sampler has seen it for ~0.7 s (these launches are not timed)
    if rank == 0:
        t_load = time.perf_counter()
        while time.perf_counter() - t_load < 0.7:
            solver.Solve(*dev_args)
            torch.cuda.synchronize(dev)
    clocks = sampler.stop() if rank == 0 else None
    sharding.barrier()
    value = world * B * args.steps / total_s
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sol)
    n_iter = sol.details.n_iter.cpu().numpy()
    status = sol.details.solve_status.cpu().numpy()
    iters_executed = float(np.where(n_iter == OPTS["max_iter"], OPTS["max_iter"], n_iter + 1).mean())
    info = nat.last_launch_info()
    sinfo = nat.last_struct_info()      # (of the device-resident launches just timed)

    # ---------------- end to end through the public API on pinned host arrays (`e2e`) ----------
    pinned = [torch.from_numpy(a).pin_memory().numpy() for a in host]
    hsolver = FCCQPBatch(n, m, nc, lcs, device=local_rank)
    hsolver.set_options(FCCQPOptionsB(**OPTS))
    hsolver.zero_copy_outputs = True     # results land in the solver's page-locked buffers, no extra host copy
    for _ in range(2):
        hsolver.Solve(*pinned)
    torch.cuda.synchronize(dev)
    sharding.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        hsolver.Solve(*pinned)           # H2D + solve + D2H, synchronous
        hsol = hsolver.GetSolution()
        zsum = float(hsol.z[:, 0].sum()) + float(hsol.details.n_iter.sum())   # host-side read of the results
    torch.cuda.synchronize(dev)
    e2e_s = sharding.max_over_ranks(time.perf_counter() - t0, dev)
    sharding.barrier()
    e2e_value = world * B * args.steps / e2e_s
    out_bytes = B * (8 * n * 2 + 8 * nc + 4 * 2 + 8 * 4)  # z/x, mu_x, mu_c, n_iter, status, 4 scalars

    # ---------------- the same, FCCQP_PRECISION_FP32_DATA (float32 problem data, FP64 arithmetic) ---------
    # NOT the headline: a different, documented precision mode (include/fccqp.h; 2e-3 bound on z) that
    # halves the PCIe bytes.  Reported next to `e2e` so the effect of the link is visible.
    f32 = None
    try:
        pinned32 = [torch.from_numpy(a.astype(np.float32)).pin_memory().numpy() for a in host]
        fsolver = FCCQPBatch(n, m, nc, lcs, device=local_rank, precision="fp32_data")
        fsolver.set_options(FCCQPOptionsB(**OPTS))
        fsolver.zero_copy_outputs = True
        for _ in range(2):
            fsolver.Solve(*pinned32)
        torch.cuda.synchronize(dev)
        sharding.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fsolver.Solve(*pinned32)
            fsol = fsolver.GetSolution()
            zsum32 = float(fsol.z[:, 0].sum())
        f32_s = sharding.max_over_ranks(time.perf_counter() - t0, dev)
        zerr = float((np.abs(fsol.z - hsol.z).max(1) / np.maximum(1.0, np.abs(hsol.z).max(1))).max())
        f32 = {"value": world * B * args.steps / f32_s, "unit": "QP/s", "ms_per_step": 1e3 * f32_s / args.steps,
               "h2d_bytes_per_step": int(sum(a.nbytes for a in pinned32)), "d2h_bytes_per_step": int(out_bytes),
               "max_rel_z_diff_vs_fp64": zerr, "stated_bound": 2e-3,
               "iteration_count_mismatches": int((fsol.details.n_iter != hsol.details.n_iter).sum())}
        del pinned32, fsolver
    except Exception as e:  # pragma: no cover
        f32 = {"error": repr(e)}
    sharding.barrier()

    # ---------------- one process, ONE call, all GPUs (fccqp_batch_solve_multi) ----------------
    # Under torchrun every rank times its own shard (above).  The C ABI can also take the whole host batch in one
    # call and split it over the devices itself (one host thread + stream set per device): rank 0 times that over
    # all `world` GPUs while the other ranks wait at the barrier.  2^15 QPs per device bound the page-locked memory.
    single_call = None
    if world > 1 and not args.no_extras:
        sharding.barrier()
        if rank == 0:
            try:
                Bs = world * (BATCH_PER_GPU // 2)
                qs = log.take(np.arange(Bs) % log.batch)
                hp = [torch.from_numpy(a).pin_memory().numpy() for a in
                      (qs.Q, qs.b, qs.A_eq, qs.b_eq, qs.friction_coeffs, qs.lb, qs.ub)]
                del qs
                ms = FCCQPBatch(n, m, nc, lcs, device=list(range(world)))
                ms.set_options(FCCQPOptionsB(**OPTS))
                ms.zero_copy_outputs = True
                ms.Solve(*hp)
                t0 = time.perf_counter()
                for _ in range(3):
                    ms.Solve(*hp)
                    zs = float(ms.GetSolution().z[:, 0].sum())
                dt = (time.perf_counter() - t0) / 3
                single_call = {"value": Bs / dt, "unit": "QP/s", "batch": Bs, "devices": world, "ms_per_call": 1e3 * dt,
                               "h2d_bytes_per_call": int(sum(a.nbytes for a in hp)),
                               "api": "FCCQPBatch(device=[0..N-1]).Solve(numpy pinned) -> fccqp_batch_solve_multi"}
                del hp, ms
            except Exception as e:  # pragma: no cover
                single_call = {"error": repr(e)}
        sharding.barrier()

    if rank != 0:
        return 0

    # ---------------- roofline + CPU baseline (rank 0) ----------------
    peaks, peak_kind = measured_peaks()
    kern_s = float(np.mean(step_ms)) * 1e-3
    alg_bytes = algorithmic_bytes_per_qp(n, m, nc) * B
    achieved = alg_bytes / kern_s / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("bytes_per_launch_at_batch_65536")
        except Exception:
            traffic = None
    flops = algorithmic_flops_per_qp(n, m, iters_executed, cold=True) * B
    fp64_nominal = 148 * 64 * 2 * 1.965e9 / 1e12  # nominal vector FP64: SMs x lanes x 2 x max clock
    fp64_peak, fp64_src = fp64_nominal, "nominal"
    try:
        tf = C.c_double(0.0)
        nat.check(nat.lib().fccqp_measure_fp64_peak(local_rank, C.byref(tf)))
        if tf.value > 0:
            fp64_peak, fp64_src = tf.value, "measured in this run: ~50 ms register-only DFMA kernel (fccqp_measure_fp64_peak)"
    except Exception:  # pragma: no cover
        pass
    # work the kernel actually EXECUTES (not the SURVEY 8d model of the dense algorithm): the structure-exploiting
    # kernel factors the reduced KKT system (Nr rows instead of n + m), every cold QP once and only the QPs that
    # iterate a second time, plus the Schur term C = A_P H^-1 A_P' and 2 Nr^2 per triangular-solve pair
    Nr = float(sinfo["rows"] if sinfo.get("used") else n + m)
    ndp = float(sum(sinfo["caps"][1:3])) if sinfo.get("used") else 0.0
    f_it = float((n_iter > 0).mean())
    per_factor = Nr ** 3 / 3.0 + m * m * ndp
    flops_exec = B * ((1.0 + f_it) * per_factor + 2.0 * Nr * Nr * (1.0 + float(n_iter.mean())))
    line = {
        "metric": METRIC, "value": value, "unit": "QP/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * total_s / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "reference walking log (2019 logged Cassie QPs, n=60 m=38 nc=12) tiled to 2^16 per GPU",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B, "n": n, "m": m, "nc": nc, "solver": OPTS,
                   "l2": "inputs (3.2 GB per step) exceed the 126 MB L2; no flush needed",
                   "launch": info, "mean_iterations_executed": iters_executed,
                   "status_counts": {str(k): int(v) for k, v in zip(*np.unique(status, return_counts=True))}},
        "e2e": {"value": e2e_value, "unit": "QP/s", "h2d_bytes_per_step": int(in_bytes),
                "d2h_bytes_per_step": int(out_bytes), "ms_per_step": 1e3 * e2e_s / args.steps,
                "api": "FCCQPBatch.Solve(numpy pinned) -> fccqp_batch_solve(FCCQP_MEM_HOST)"},
        "e2e_fp32_data": f32,
        "e2e_single_call_all_gpus": single_call,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                     "frac": achieved / peaks.get("hbm_gbs"), "traffic": traffic, "peak_source": peak_kind,
                     "kernel": "fccqp_struct_kernel" if sinfo.get("used") else "fccqp_solve_kernel", "kernel_ms": 1e3 * kern_s,
                     "note": "latency/FP64-bound kernel: HBM fraction is low by construction; see fp64"},
        "roofline_fp64": {"achieved_tflops": flops / kern_s / 1e12, "peak_tflops": fp64_peak, "peak_source": fp64_src,
                          "peak_tflops_nominal": fp64_nominal, "frac": flops / kern_s / 1e12 / fp64_peak,
                          "flops_model": "SURVEY 8d (the dense algorithm): 2 x N^3/3 + 2 N^2 x iterations_executed per cold QP",
                          "executed_tflops": flops_exec / kern_s / 1e12, "frac_executed": flops_exec / kern_s / 1e12 / fp64_peak,
                          "executed_model": "counted: (1 + iterating fraction) x (Nr^3/3 + m^2 ndp) + 2 Nr^2 x (1 + mean n_iter), "
                                            "Nr = KKT rows factored per QP",
                          "kkt_rows_factored": Nr, "kkt_rows_dense": float(n + m), "iterating_fraction": f_it},
        "structure": sinfo,
        "latency": {"p50_ms_per_batch_launch": float(np.median(step_ms))},
    }
    # p50 latency of one warm Solve through the drop-in FCCQP object (fcc_qp_test.py loop)
    try:
        from fcc_qp_b200 import FCCQP, FCCQPOptions
        s1 = FCCQP(n, m, nc, lcs)
        o = FCCQPOptions(); o.max_iter, o.rho, o.eps_fcone, o.eps_bound = (OPTS[k] for k in ("max_iter", "rho", "eps_fcone", "eps_bound"))
        s1.set_options(o)
        lat = []
        for i in range(200):
            s1.set_warm_start(i > 0)
            q = log.qp(i)
            t1 = time.perf_counter()
            s1.Solve(q["Q"], q["b"], q["A_eq"], q["b_eq"], q["friction_coeffs"], q["lb"], q["ub"])
            s1.GetSolution()
            lat.append(time.perf_counter() - t1)
        line["latency"]["p50_us_single_solve_dropin"] = float(np.median(lat[20:]) * 1e6)
    except Exception as e:  # pragma: no cover
        line["latency"]["single_solve_error"] = repr(e)
    if world == 1:
        try:
            rate, cores, kind, secs = cpu_reference_run(log, 2019)
            sample = int(min(B, max(2019, rate * 12.0)))
            # ~10 s of all-core CPU work: the sample (at most the bench batch itself) solved repeatedly
            reps = int(min(12, max(1, round(10.0 * rate / sample))))
            tot = 0.0
            for _ in range(reps):
                rate_i, cores, kind, secs = cpu_reference_run(log, sample)
                tot += secs
            rate = reps * sample / tot
            line["cpu_baseline"] = {"value": rate, "unit": "QP/s", "cores": cores, "kind": kind,
                                    "sample": f"first {sample} QPs of the same tiled log, cold, solved {reps}x, {tot:.1f} s"}
        except Exception as e:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "unit": "QP/s", "cores": 0, "kind": "port", "sample": repr(e)}
        if not args.no_extras:
            line["cpu_baseline_variants"] = cpu_baseline_variants(log, 4038)
            del dev_args, pinned
            torch.cuda.empty_cache()
            line["shapes"] = shape_extras(dev)
    emit(line)
    return 0


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the process's real stdout."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # Only the JSON line may reach stdout: library banners (e.g. "NCCL version ..." at communicator
    # creation) are written to file descriptor 1 behind Python's back, so fd 1 is pointed at stderr for
    # the whole run and the line goes to a private duplicate of the original stdout.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the extra keys (other shapes, CPU baseline variants)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's solution arrays to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU solver (--impl ours)")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
