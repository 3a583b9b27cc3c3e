"""compute-sanitizer is closed on this pool: the kernels that alias shared-memory boards on purpose (csrc/sls_t16.cu, csrc/sls_p16.cu)
check themselves.
Builds libtss with -DTSS_CHECKED (every shared-memory access of the step loop verified: loads inside the CTA's Smem block, stores
in a row of the grid of the board they mean) into build/libtss_checked.so; run the trajectory / warm-start / optimum tests and a
randomized campaign against it with TSS_LIB pointing there, then read tss_debug_smem_violations().

    python profiles/checked_build.py build          # here (nvcc, no GPU needed)
    TSS_LIB=$PWD/build/libtss_checked.so python profiles/checked_build.py run     # on the GPU box
"""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "build", "libtss_checked.so")
if sys.argv[1:] == ["build"]:
    from timberborn_support_solver_b200 import build as B
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    cmd = [os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), *B.NVCC_FLAGS, "-DTSS_CHECKED", "-o", OUT, *[os.path.join(B.CSRC, s) for s in B.SOURCES]]
    subprocess.check_call(cmd, cwd=B.CSRC)
    print(OUT)
else:
    assert os.environ.get("TSS_LIB") == OUT, "run with TSS_LIB=" + OUT
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import oracle.oracle as O
    import timberborn_support_solver_b200 as T
    from conftest import synth_terrain
    lib = T.load()
    assert lib.tss_debug_smem_violations() == 0, "not a checked build"
    eng = T.Engine(0)
    rng = np.random.default_rng(7)
    runs = 0
    for case in range(int(sys.argv[2]) if len(sys.argv) > 2 else 600):
        w, h = int(rng.integers(1, 27)), int(rng.integers(1, 17))
        dens = float(rng.choice([0.3, 0.6, 0.85, 1.0]))
        grid = synth_terrain(w, h, seed=int(rng.integers(1, 1000)), t=int(rng.integers(0, 1000)), density_q24=int(dens * (1 << 24)))
        if grid.sum() == 0:
            continue
        n_chains, seed = int(rng.integers(1, 300)), int(rng.integers(0, 1 << 30))
        epochs = [(int(rng.integers(1, 500)), 1 << 20, 0) for _ in range(int(rng.integers(1, 3)))]
        warm = None
        if rng.random() < 0.4:      # dense warm starts drive all five count planes and rows at the grid's edge
            warm = np.zeros((n_chains, 32, 32), np.uint8)
            warm[:, :h, :w] = rng.random((n_chains, h, w)) < rng.choice([0.1, 0.5, 1.0])
        want = None
        for kernel in (T.KERNEL_THREAD, T.KERNEL_PAIR) if w <= 16 else (T.KERNEL_THREAD,):   # row pairs: grids of at most 16x16
            s = eng.search(T.WorldGrid(grid), seed=seed, n_chains=n_chains, kernel=kernel)
            if warm is not None:
                s.write_chains((warm.astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(2, dtype=np.uint32))
            for steps, _, target in epochs:
                s.run(steps, target)
            got = s.read_chains()
            if n_chains <= 24:          # and the results are still the model's
                want = want or O.sls_model(grid, n_chains, epochs, seed=seed, init_S=warm)
                assert np.array_equal(got["k"], want["k"]) and np.array_equal(got["best"], want["best"]) and np.array_equal(got["scored"], want["scored"])
            s.close()
            runs += 1
    g16 = T.WorldGrid(np.ones((16, 16), np.uint8))
    for kernel in (T.KERNEL_THREAD, T.KERNEL_PAIR):
        s = eng.search(g16, seed=1, kernel=kernel)        # the bench's configuration: the device filled with chains
        for _ in range(3):
            s.run(2048, 0)
        assert s.best_count() == 15
        s.close()
    v = lib.tss_debug_smem_violations()
    print(f"checked build: {runs} randomized runs of sls_t16_kernel (grids up to 26x16) and sls_p16_kernel (grids up to 16x16), 1-300 chains, "
          f"dense warm starts, + the bench configuration on both: {v} shared-memory violations")
    assert v == 0
