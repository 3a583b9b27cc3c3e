"""Builds timberborn_support_solver_b200/libtss.so (the C-ABI library of include/tss.h) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libtss.so")
SOURCES = ["engine.cu", "eval.cu", "eval_thread.cu", "cnf.cu", "sls.cu", "sls_h16.cu", "sls_t16.cu", "sls_p16.cu", "sls_multi.cu", "lns.cu", "lns_placements.cu", "greedy.cu", "lb.cu", "lp.cu", "lp_big.cu", "comm.cu", "peaks.cu", "capi_host.cpp", "host_model.cpp", "instance.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math",
              "-Xcompiler", "-fPIC,-Wall,-Wno-unknown-pragmas", "-shared", "-cudart", "static", "-ldl"]


TOOLS = os.path.join(HERE, "tools")
REPL = os.path.join(HERE, "tss_repl")   # the C++ driver that mirrors the REPL's `solve` over the C ABI (tools/tss_repl.cpp)


def needs_build() -> bool:
    if not os.path.exists(OUT) or not os.path.exists(REPL):
        return True
    t = min(os.path.getmtime(OUT), os.path.getmtime(REPL))
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(TOOLS, f) for f in os.listdir(TOOLS)] + [os.path.join(HERE, "..", "include", "tss.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, *NVCC_FLAGS, *(["-Xptxas", "-v"] if verbose else []), "-o", OUT, *[os.path.join(CSRC, s) for s in SOURCES]]
    subprocess.check_call(cmd, cwd=CSRC)
    subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-Wall", "-o", REPL, os.path.join(TOOLS, "tss_repl.cpp"),
                           "-L" + HERE, "-ltss", "-Wl,-rpath,$ORIGIN"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
