"""The C restatement (oracle/fccqp_oracle.c) with the rho each solve ended with recorded -- test infrastructure of the
per-lane rho tests (tests/test_rho_lanes.py, tests/test_gpu_rho_lanes.py).

Adaptive rho moves rho inside do_admm and drops it at exit; the per-lane rho of the batched solve hands that value to the
next warm solve, so its oracle has to report it.  The restatement's source is compiled here, into a directory the caller
gives, with the flags of oracle/Makefile and three additions that change no arithmetic: a static `g_rho_last`, set to the
options' rho before ADMM and to do_admm's final rho at its end, and `fccqp_oracle_last_rho()` returning it.  The
checked-in oracle stays as it is.  One solver object at a time (the value is process-wide in this library).
"""
import ctypes as C
import os
import subprocess

import oracle

SRC = os.path.join(os.path.dirname(oracle.__file__), "fccqp_oracle.c")
# (anchor in the restatement, replacement); each anchor must occur exactly once
EDITS = [
    ("  if (!equality_constrained) do_admm(o, b, mu, lb, ub);",
     "  g_rho_last = o->rho;   /* (an equality-constrained QP runs no ADMM) */\n"
     "  if (!equality_constrained) do_admm(o, b, mu, lb, ub);"),
    ("  free(lcbar_prev);\n}", "  free(lcbar_prev);\n  g_rho_last = rho;\n}"),
]


def build(outdir) -> str:
    src = open(SRC).read()
    for old, new in EDITS:
        assert src.count(old) == 1, f"anchor not found once in {SRC}: {old!r}"
        src = src.replace(old, new)
    src = "static double g_rho_last;\n" + src + "\ndouble fccqp_oracle_last_rho(void) { return g_rho_last; }\n"
    c = os.path.join(str(outdir), "fccqp_oracle_rho.c")
    so = os.path.join(str(outdir), "libfccqp_oracle_rho.so")
    with open(c, "w") as f:
        f.write(src)
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-std=c11", "-fPIC", "-shared", "-pthread",
                           "-I", os.path.dirname(SRC), "-o", so, c, "-lm"])
    return so


def load(outdir) -> oracle.Oracle:
    """An Oracle("port") over the library above (same ctypes set-up), with .last_rho() added."""
    so = build(outdir)
    saved = oracle._PORT_SO
    oracle._PORT_SO = so           # (Oracle.__init__ loads the port library from this path)
    try:
        orc = oracle.Oracle("port")
    finally:
        oracle._PORT_SO = saved
    orc.lib.fccqp_oracle_last_rho.restype = C.c_double
    orc.last_rho = lambda: float(orc.lib.fccqp_oracle_last_rho())
    return orc
