"""Where a step of sls_p16_kernel spends its clocks, at the bench's shape (rect 16x16, 1x1 supports, the default portfolio of
SMs x 3 x 128 chains, 4 096-step epochs).  The phase-profiling build (-DTSS_SLS_PROF, sls_thread.cuh) reads clock64() between
the parts of every step and sums the differences per thread; this prints them per chain step, i.e. the clocks a warp spends
on one step, split into: the removal scan, the removal's swap and flip, the addition's fetch and tabu window, the 25
candidates and the decode, the addition's flip, and the loop frame.  The marks cost registers and issue slots of their own, so
compare builds by their totals here and by bench.py for rates.

    python profiles/sls_phases.py build OUT.so           # here (nvcc, no GPU needed): libtss with -DTSS_SLS_PROF
    python profiles/sls_phases.py run LABEL=LIB [...]    # on the GPU: one process per build, all in one run
"""
import ctypes
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PHASES = ["removal scan", "removal swap + flip", "fetch + tabu window", "candidates + decode", "addition flip", "loop frame"]
WARM, EPOCHS, EPOCH_STEPS = 3, 5, 4096


def one():
    import numpy as np
    import timberborn_support_solver_b200 as T
    lib = T.load()
    read = lib.tss_debug_sls_p16_phases   # only a -DTSS_SLS_PROF build has it
    read.argtypes, read.restype = [ctypes.POINTER(ctypes.c_ulonglong)], ctypes.c_int
    out = (ctypes.c_ulonglong * (len(PHASES) + 1))()
    eng = T.Engine(0)
    s = eng.search(T.WorldGrid(np.ones((16, 16), np.uint8)), seed=1, kernel=T.KERNEL_PAIR)
    for _ in range(WARM):
        s.run(EPOCH_STEPS, 0)
    s.best_count()
    assert read(out) == len(PHASES), "phase totals not readable"
    t0 = time.perf_counter()
    for _ in range(EPOCHS):
        s.run(EPOCH_STEPS, 0)
    best = s.best_count()
    ms = (time.perf_counter() - t0) * 1e3 / EPOCHS
    assert read(out) == len(PHASES)
    steps = out[len(PHASES)]
    cyc = [out[i] / steps for i in range(len(PHASES))]
    tot = sum(cyc)
    print(f"  chains {s.n_chains}, {EPOCHS} epochs x {EPOCH_STEPS} steps, {steps} chain steps, best {best}, {ms:.2f} ms per epoch (host clock, profiled build)")
    for name, c in zip(PHASES, cyc):
        print(f"  {name:24s} {c:8.1f} clocks per step  {100 * c / tot:5.1f} %")
    print(f"  {'total':24s} {tot:8.1f} clocks per step")
    s.close()


def main():
    if sys.argv[1] == "build":
        from timberborn_support_solver_b200 import build as B
        out = os.path.abspath(sys.argv[2])
        os.makedirs(os.path.dirname(out), exist_ok=True)
        cmd = [os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), *B.NVCC_FLAGS, "-DTSS_SLS_PROF", "-o", out, *[os.path.join(B.CSRC, s) for s in B.SOURCES]]
        subprocess.check_call(cmd, cwd=B.CSRC)
        print(out)
    elif sys.argv[1] == "one":
        one()
    else:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
        print("name, power.limit, clocks.max.sm, clocks.sm:", smi.strip().split("\n")[0])
        for label, lib in (b.split("=", 1) for b in sys.argv[2:]):
            print(f"{label}: {lib}", flush=True)
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "one"], env=dict(os.environ, TSS_LIB=os.path.abspath(lib)), cwd=ROOT)


if __name__ == "__main__":
    main()
