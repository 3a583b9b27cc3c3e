"""The row-pair kernel's support cache (csrc/sls_p16.cu: the first CAP site-list entries of a chain and their reach
windows in shared memory, the rest in the global list).  Lists that start at, just below and just above CAP, lists of
every cell of the grid, and lists that grow past CAP and shrink back below it within one epoch must all replay the CPU
model and the flat port bit for bit; and the cache must still leave three 128-chain CTAs resident per SM."""
import os
import re
import subprocess

import numpy as np
import pytest

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import synth_terrain
from test_sls_row_pairs import BIG, eng, terrain, unpack  # noqa: F401  (eng is a fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "timberborn_support_solver_b200", "csrc")
with open(os.path.join(CSRC, "sls_p16.cu")) as _f:
    CAP = int(re.search(r"constexpr int CAP = (\d+);", _f.read()).group(1))


def grid_of(fixtures, name):
    if name == "random16x16":      # dense random terrain: its optimum lies below CAP, its first complete layouts above
        return synth_terrain(16, 16, seed=5, t=4, density_q24=int(0.9 * (1 << 24)))
    return terrain(fixtures, name)


def rows_of(init):
    return (init.astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(2, dtype=np.uint32)


def replay(eng, grid, n_chains, epochs, seed, offset, init):  # noqa: F811
    """runs the pair kernel from `init` and checks it against the CPU model and the flat port"""
    s = eng.search(T.WorldGrid(grid), seed=seed, n_chains=n_chains, chain_offset=offset, kernel=T.KERNEL_PAIR)
    assert s.kernel_variant() == T.KERNEL_PAIR
    if init is not None:
        s.write_chains(rows_of(init))
    flips0 = eng.stats()["sls_flips"]
    for steps, _, target in epochs:
        s.run(steps, target)
    got = s.read_chains()
    flips = eng.stats()["sls_flips"] - flips0
    s.close()
    want = O.sls_model(grid, n_chains, epochs, seed=seed, chain_offset=offset, share_bound=True, init_S=init)
    flat = O.sls_flat(grid, n_chains, epochs, seed=seed, chain_offset=offset, share_bound=True, init_S=init, threads=2)
    for key in ("k", "best", "step", "scored"):
        assert np.array_equal(got[key], want[key]), key
        assert np.array_equal(flat[key], want[key]), key
    assert np.array_equal(unpack(got["S"]), want["S"]) and np.array_equal(unpack(got["bestS"]), want["bestS"])
    assert np.array_equal(flat["S"], want["S"])
    assert flips == int(flat["flips"].sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rect16x16", "ex3", "random16x16"])
def test_warm_starts_around_cap_bit_exact(eng, fixtures, name):  # noqa: F811
    """Chains start with CAP-1, CAP, CAP+1 supports or one on every cell of the grid (256 on a 16x16 grid; supports under
    non-ceiling tiles too), so list entries sit on both sides of CAP from the first step and the drops move global
    entries into cached slots."""
    grid = grid_of(fixtures, name)
    h, w = grid.shape
    counts = [CAP - 1, CAP, CAP + 1, h * w]
    n_chains = 40
    rng = np.random.default_rng(12)
    init = np.zeros((n_chains, 32, 32), np.uint8)
    for c in range(n_chains):
        n = counts[c % 4]
        cells = rng.choice(h * w, n, replace=False)
        init[c, cells // w, cells % w] = 1
    assert sorted({int(init[c].sum()) for c in range(n_chains)}) == sorted(set(counts))
    replay(eng, grid, n_chains, [(150, BIG, -1), (400, BIG, -1)], seed=6, offset=11, init=init)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rect16x16", "ex3", "random16x16"])
def test_list_crosses_cap_both_ways_in_one_epoch(eng, fixtures, name):  # noqa: F811
    """Lists that grow past CAP (additions into the global list) and then shrink below it (removals that pull global
    entries back into the cache) inside one launch.  rect 16x16 and the random terrain start empty and overshoot to
    20-24 supports before their first complete layout; ex3 starts from CAP-1 supports crowded into its three leftmost
    columns, so it has to add several before the layout is complete."""
    grid = grid_of(fixtures, name)
    n_chains, seed, steps = 40, 9, 500
    init = None
    if name == "ex3":
        rng = np.random.default_rng(1)
        init = np.zeros((n_chains, 32, 32), np.uint8)
        for c in range(n_chains):
            cells = rng.choice(grid.shape[0] * 3, CAP - 1, replace=False)
            init[c, cells // 3, cells % 3] = 1
    # the model's k after the first s steps of the same epoch: some chain has to be above CAP and later below it
    ks = np.array([O.sls_model(grid, n_chains, [(s, BIG, -1)], seed=seed, init_S=init)["k"] for s in (5, 10, 20, 30, 40, 60, 120, 300, steps)])
    crossed = [c for c in range(n_chains) if (ks[:, c] > CAP).any() and (ks[np.argmax(ks[:, c] > CAP):, c] < CAP).any()]
    assert len(crossed) >= n_chains // 4, (name, ks.max(1), ks.min(1))
    replay(eng, grid, n_chains, [(steps, BIG, -1)], seed=seed, offset=0, init=init)


@pytest.mark.gpu
def test_three_ctas_per_sm(tmp_path):
    """cudaOccupancyMaxActiveBlocksPerMultiprocessor for the kernel as the library launches it (128 threads, its whole
    shared-memory block): exactly 3, so the default portfolio of 3 x 128 chains per SM fills every SM evenly."""
    from timberborn_support_solver_b200 import build as B
    src = tmp_path / "occupancy.cu"
    src.write_text('#include <cstdio>\n#include "sls_p16.cu"\nint main() {\n'
                   "    using namespace tss::slsp;\n"
                   "    if (cudaFuncSetAttribute(sls_p16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES) != cudaSuccess) return 2;\n"
                   "    int n = 0;\n"
                   "    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, sls_p16_kernel, NT, SMEM_BYTES) != cudaSuccess) return 3;\n"
                   '    printf("%d %zu\\n", n, SMEM_BYTES);\n    return 0;\n}\n')
    exe = tmp_path / "occupancy"
    flags = [f for f in B.NVCC_FLAGS if f not in ("-shared",)]
    subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), *flags, "-I", CSRC, "-o", str(exe), str(src)], check=True, cwd=tmp_path)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    ctas, smem = int(out[0]), int(out[1])
    assert ctas == 3, (ctas, smem)
    assert smem > 64 * 1024          # the cache is in the block: no padding left to decide the occupancy
