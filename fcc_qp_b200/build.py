"""In-tree build of the native pieces (run by ``__graft_entry__.build()``).

* ``libfccqp_b200.so``  -- CUDA kernels + C ABI (``csrc/fccqp_capi.cu``), nvcc, sm_100a only.
* ``fcc_qp_solver*.so`` -- pybind11 module with the reference's class names
  (``csrc/pybind_module.cpp`` over the header-only ``include/fcc_qp.hpp``), g++, links the C ABI library.

Everything lands next to this file so that it travels with the repository
snapshot to the GPU box; nothing is JIT-compiled at import time.
"""
from __future__ import annotations

import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libfccqp_b200.so")
NVCC_ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _stale(target: str, sources) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd, verbose):
    if verbose:
        print("+", " ".join(cmd), flush=True)
    subprocess.check_call(cmd)


def pybind_target() -> str:
    return os.path.join(HERE, "fcc_qp_solver" + sysconfig.get_config_var("EXT_SUFFIX"))


def build_cuda(force=False, verbose=False, extra=()):
    srcs = [os.path.join(CSRC, f) for f in ("fccqp_capi.cu", "fccqp_kernel.cuh", "fccqp_struct.cuh", "fccqp_warp.cuh", "fccqp_polish.cuh")] + \
           [os.path.join(ROOT, "include", "fccqp.h")]
    if force or _stale(LIB, srcs):
        nvcc = os.environ.get("NVCC", "nvcc")
        # FCCQP_DEV=1 compiles the developer instrumentation in (FCCQP_PROFILE phase counters); the
        # production build leaves it out: the hot loops have to fit the instruction cache.
        dev = ["-DFCCQP_DEV"] if os.environ.get("FCCQP_DEV") else []
        _run([nvcc, *NVCC_ARCH, "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
              *dev, *extra, "-o", LIB, os.path.join(CSRC, "fccqp_capi.cu")], verbose)
    return LIB


def build_pybind(force=False, verbose=False):
    import pybind11
    tgt = pybind_target()
    srcs = [os.path.join(CSRC, "pybind_module.cpp"), os.path.join(ROOT, "include", "fcc_qp.hpp"),
            os.path.join(ROOT, "include", "fccqp.h"), LIB]
    if force or _stale(tgt, srcs):
        cxx = os.environ.get("CXX", "g++")
        _run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
              "-I", pybind11.get_include(), "-I", sysconfig.get_paths()["include"],
              "-I", os.path.join(ROOT, "include"),
              os.path.join(CSRC, "pybind_module.cpp"),
              "-L", HERE, "-lfccqp_b200", "-Wl,-rpath,$ORIGIN", "-o", tgt], verbose)
    return tgt


def build_cpp_dropin(force=False, verbose=False, eigen="/root/reference/eigen"):
    """tests/cpp/dropin_main: a caller written against the reference's Eigen-typed C++ surface, compiled
    against include/fcc_qp.hpp.  Needs Eigen headers (the reference's vendored copy; not on the GPU box,
    where the prebuilt binary is used).  Returns the binary path or None."""
    src = os.path.join(ROOT, "tests", "cpp", "dropin_main.cpp")
    tgt = os.path.join(ROOT, "tests", "cpp", "dropin_main")
    if not os.path.isdir(eigen) or not os.path.exists(src):
        return tgt if os.path.exists(tgt) else None
    if force or _stale(tgt, [src, os.path.join(ROOT, "include", "fcc_qp.hpp"), os.path.join(ROOT, "include", "fccqp.h"), LIB]):
        cxx = os.environ.get("CXX", "g++")
        _run([cxx, "-std=c++17", "-O1", "-w", "-I", eigen, "-I", os.path.join(ROOT, "include"), src,
              "-L", HERE, "-lfccqp_b200", "-Wl,-rpath,$ORIGIN/../../fcc_qp_b200", "-o", tgt], verbose)
    return tgt


def build_all(force=False, verbose=False):
    build_cuda(force, verbose)
    build_pybind(force, verbose)
    build_cpp_dropin(force, verbose)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose=True)
