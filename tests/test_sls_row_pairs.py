"""The row-pair thread-per-chain SLS kernel (TSS_KERNEL_PAIR, csrc/sls_p16.cu: one chain per thread, two grid rows per
32-bit word, grids of at most 16x16) against the CPU model, the flat CPU port and the one-row-per-word kernel (t16).
Its windows keep the spec's clamped anchor and come in two row-slot alignments, so the shapes below cover even and odd
heights (both alignments and a last half-filled pair), the left and right edges, one-row and one-column grids."""
import os
import re

import numpy as np
import pytest

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import synth_terrain

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIG = 1 << 20


def unpack(rows):
    return ((rows[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8)


@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def terrain(fixtures, name):
    w, h = (int(s) for s in re.findall(r"\d+", name)[-2:]) if name.startswith(("rect", "synth")) else (0, 0)
    if name.startswith("rect"):
        return np.ones((h, w), np.uint8)
    if name.startswith("synth"):
        return synth_terrain(w, h, seed=3, t=w * 17 + h)
    return {"ex1": fixtures["ex1"].T.copy(), "ex3": fixtures["ex3"]}[name]


# w x h: rect 16x16 and the fixtures; 16x9, 13x15 (odd heights: the last pair is half filled), 9x12, 13x16, one row, one
# column, 3x3, and synthetic terrains (70 % ceiling) of both parities
TRAJECTORY_CASES = ["rect16x16", "ex1", "ex3", "rect16x9", "rect9x12", "rect13x16", "rect16x1", "rect1x16", "rect3x3",
                    "synth16x16", "synth16x15", "synth11x7", "synth13x15"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", TRAJECTORY_CASES)
def test_pair_kernel_trajectories_bit_exact(eng, fixtures, name):
    grid = terrain(fixtures, name)
    n_chains, offset, seed = 150, 100, 7          # two CTAs, the second one partially filled
    epochs = [(50, BIG, 0), (300, BIG, 0), (1000, BIG, 0)]
    s = eng.search(T.WorldGrid(grid), seed=seed, n_chains=n_chains, chain_offset=offset, kernel=T.KERNEL_PAIR)
    assert s.kernel_variant() == T.KERNEL_PAIR
    flips0 = eng.stats()["sls_flips"]
    for steps, _, target in epochs:
        s.run(steps, target)
    got = s.read_chains()
    want = O.sls_model(grid, n_chains, epochs, seed=seed, chain_offset=offset, share_bound=True)
    flat = O.sls_flat(grid, n_chains, epochs, seed=seed, chain_offset=offset, share_bound=True, threads=2)
    for key in ("k", "best", "step", "scored"):
        assert np.array_equal(got[key], want[key]), key
        assert np.array_equal(flat[key], want[key]), key
    assert np.array_equal(unpack(got["S"]), want["S"]) and np.array_equal(unpack(got["bestS"]), want["bestS"])
    assert np.array_equal(flat["S"], want["S"]) and np.array_equal(flat["bestS"], want["bestS"])
    assert eng.stats()["sls_flips"] - flips0 == int(flat["flips"].sum())
    assert s.best_count() == int(want["best"].min())
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rect16x16", "synth16x15", "ex3"])
def test_pair_kernel_dense_warm_starts_bit_exact(eng, fixtures, name):
    """Dense starts drive the cover counts through all five count planes (a pair word carries two rows' carries)."""
    grid = terrain(fixtures, name)
    h, w = grid.shape
    n_chains = 40
    rng = np.random.default_rng(5)
    init = np.zeros((n_chains, 32, 32), np.uint8)
    for c in range(n_chains):
        dens = [1.0, 0.5, 0.25, 0.1][c % 4]
        init[c, :h, :w] = (rng.random((h, w)) < dens) & ((grid != 0) | (c % 8 >= 4))     # some supports under non-ceiling tiles
    rows = (init.astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(2, dtype=np.uint32)
    epochs = [(120, BIG, -1), (200, BIG, -1)]
    s = eng.search(T.WorldGrid(grid), seed=4, n_chains=n_chains, chain_offset=7, kernel=T.KERNEL_PAIR)
    s.write_chains(rows)
    for steps, _, target in epochs:
        s.run(steps, target)
    got = s.read_chains()
    want = O.sls_model(grid, n_chains, epochs, seed=4, chain_offset=7, share_bound=True, init_S=init)
    for key in ("k", "best", "step", "scored"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(unpack(got["S"]), want["S"]) and np.array_equal(unpack(got["bestS"]), want["bestS"])
    s.close()


@pytest.mark.gpu
def test_pair_kernel_degenerate_terrains(eng):
    """No ceiling, a single tile, a 16-wide one-row corridor, isolated tiles."""
    cases = [np.zeros((4, 7), np.uint8), np.pad(np.ones((1, 1), np.uint8), ((2, 3), (4, 1))), np.ones((1, 16), np.uint8),
             (np.indices((16, 16)).sum(0) % 2 == 0).astype(np.uint8) * (np.indices((16, 16))[0] % 2 == 0)]
    for grid in cases:
        grid = np.ascontiguousarray(grid, np.uint8)
        epochs = [(30, BIG, 0), (200, BIG, 0)]
        s = eng.search(T.WorldGrid(grid), seed=2, n_chains=33, chain_offset=3, kernel=T.KERNEL_PAIR)
        for steps, _, target in epochs:
            s.run(steps, target)
        got = s.read_chains()
        want = O.sls_model(grid, 33, epochs, seed=2, chain_offset=3, share_bound=True)
        for key in ("k", "best", "step", "scored"):
            assert np.array_equal(got[key], want[key]), (key, grid.shape)
        assert np.array_equal(unpack(got["S"]), want["S"]) and np.array_equal(unpack(got["bestS"]), want["bestS"])
        assert s.best_count() == int(want["best"].min())
        s.close()


@pytest.mark.gpu
def test_pair_kernel_long_run_split_at_32768_steps(eng):
    grid = np.ones((8, 8), np.uint8)
    epochs = [(40000, BIG, -1)]
    want = O.sls_model(grid, 40, epochs, seed=11, chain_offset=0, share_bound=True)
    s = eng.search(T.WorldGrid(grid), seed=11, n_chains=40, kernel=T.KERNEL_PAIR)
    s.run(40000, -1)
    got = s.read_chains()
    for key in ("k", "best", "step", "scored"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(unpack(got["S"]), want["S"])
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["rect16", "ex3", "random16x16", "random12x9-dense"])
def test_pair_kernel_agrees_with_t16_at_scale(eng, fixtures, case):
    """Thousands of chains x tens of thousands of steps (too many for the CPU model): chain states, counters and bounds
    after every epoch are those of the one-row-per-word kernel."""
    grid = {"rect16": np.ones((16, 16), np.uint8), "ex3": fixtures["ex3"], "random16x16": synth_terrain(16, 16, seed=7, t=1),
            "random12x9-dense": synth_terrain(12, 9, seed=8, t=2, density_q24=int(0.93 * (1 << 24)))}[case]
    n_chains = 2048 + 77
    runs = {}
    for kernel in (T.KERNEL_THREAD, T.KERNEL_PAIR):
        s = eng.search(T.WorldGrid(grid), seed=21, n_chains=n_chains, chain_offset=5, kernel=kernel)
        assert s.kernel_variant() == kernel
        flips0 = eng.stats()["sls_flips"]
        snaps = []
        for steps in (700, 6000, 40000):
            s.run(steps, 0)
            snaps.append((s.best_count(), s.global_best()))
        runs[kernel] = (snaps, s.read_chains(), eng.stats()["sls_flips"] - flips0)
        s.close()
    (ref_snaps, ref, ref_flips), (snaps, st, flips) = runs[T.KERNEL_THREAD], runs[T.KERNEL_PAIR]
    assert snaps == ref_snaps and flips == ref_flips
    for key in ("S", "bestS", "k", "best", "step", "scored"):
        assert np.array_equal(st[key], ref[key]), key


@pytest.mark.gpu
def test_pair_kernel_selection(eng, fixtures):
    for grid in (np.ones((16, 17), np.uint8), np.ones((17, 16), np.uint8)):       # 17 wide, 17 tall
        with pytest.raises(T.TssError):
            eng.search(T.WorldGrid(grid), n_chains=8, kernel=T.KERNEL_PAIR)
    s = eng.search(T.WorldGrid(np.ones((16, 16), np.uint8)))                       # auto, default chains: the device filled
    assert s.kernel_variant() == T.KERNEL_PAIR
    assert s.n_chains == eng.device_info()["sm_count"] * 3 * 128
    s.close()
    s = eng.search(T.WorldGrid(np.ones((16, 16), np.uint8)), kernel=T.KERNEL_THREAD)   # pinned t16 still runs t16
    assert s.kernel_variant() == T.KERNEL_THREAD
    s.close()
    s = eng.search(T.WorldGrid(fixtures["ex2"]))                                    # 21 wide: one row per word
    assert s.kernel_variant() == T.KERNEL_THREAD
    s.close()


def test_pair_kernel_constant_in_every_binding():
    with open(os.path.join(ROOT, "include", "tss.h")) as f:
        assert re.search(r"#define TSS_KERNEL_PAIR 4\b", f.read())
    with open(os.path.join(ROOT, "rust", "tss-sys", "src", "lib.rs")) as f:
        assert re.search(r"pub const TSS_KERNEL_PAIR: i32 = 4;", f.read())
    assert T.KERNEL_PAIR == 4
    from timberborn_support_solver_b200 import build as B
    assert "sls_p16.cu" in B.SOURCES
