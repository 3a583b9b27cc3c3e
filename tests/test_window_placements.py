"""The window-decomposed placement search (TSS_KERNEL_WINDOW_PLACEMENTS, csrc/lns_placements.cu driving
sls_multi_kernel<false, true>) on grids larger than 32x32: its scalar replay (tests/window_model.py) keeps the global
layout valid phase after phase, and the GPU follows the replay bit for bit."""
import os
import re

import numpy as np
import pytest

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import synth_terrain
from window_model import lns_placements_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUI_WEIGHTS = {(1, 1): 3, (1, 3): 2, (3, 3): 4, (5, 5): 7}
RANDOM_SET = [(1, 1), (2, 3), (2, 2), (1, 4), (4, 4)]


def keys_of(defs):
    """The engine's dims keys: both orientations of every def in defs order, unflipped first, duplicates dropped
    -> (effective dims per key, (def_w, def_h, rotated) per key)."""
    dims, proto = [], []
    for w, h in defs:
        for rot in (0, 1):
            d = (h, w) if rot else (w, h)
            if d not in dims:
                dims.append(d)
                proto.append((w, h, rot))
    return dims, proto


def key_costs(dims, weights):
    """cost of a platform = sum of the weights of every def that fits inside its def (platform_layout.rs:174-183)"""
    if not weights:
        return [1] * len(dims)
    canon = lambda w, h: (min(w, h), max(w, h))
    return [sum(v for d, v in weights.items() if canon(*d)[0] <= canon(w, h)[0] and canon(*d)[1] <= canon(w, h)[1]) for w, h in dims]


def check_valid(grid, dims, proto, layout):
    v = O.validate(grid, [(x, y, *proto[k]) for x, y, k in layout])
    assert v.is_valid, (int(v.unsupported.sum()), v.overlapping[:3], v.out_of_bounds[:3])
    h, w = grid.shape
    for x, y, k in layout:
        assert 0 <= k < len(dims) and x + dims[k][0] <= w and y + dims[k][1] <= h


def random_start(grid, dims, proto, seed):
    """A random valid layout: random non-overlapping placements, then a 1x1 on every ceiling tile left unsupported."""
    h, w = grid.shape
    rng = np.random.default_rng(seed)
    occ = np.zeros((h, w), bool)
    out = []
    for _ in range(w * h // 12):
        k = int(rng.integers(1, len(dims)))
        pw, ph = dims[k]
        x, y = int(rng.integers(0, w - pw + 1)), int(rng.integers(0, h - ph + 1))
        if not occ[y:y + ph, x:x + pw].any():
            occ[y:y + ph, x:x + pw] = True
            out.append((x, y, k))
    uns = O.validate(grid, [(x, y, *proto[k]) for x, y, k in out]).unsupported.astype(bool)
    out += [(int(x), int(y), 0) for y, x in zip(*np.nonzero(uns & ~occ))]
    return out


@pytest.mark.parametrize("shape", [(48, 40), (70, 33), (33, 90)])
@pytest.mark.parametrize("start_kind", ["all-1x1", "random"])
def test_model_keeps_the_global_layout_valid(shape, start_kind):
    w, h = shape
    grid = synth_terrain(w, h, seed=2, t=w + h)
    dims, proto = keys_of(O.PLATFORMS_DEFAULT)
    if start_kind == "all-1x1":
        start = [(int(x), int(y), 0) for y, x in zip(*np.nonzero(grid))]
    else:
        start = random_start(grid, dims, proto, seed=w * h)
    check_valid(grid, dims, proto, start)
    r = lns_placements_model(grid, dims, [1] * len(dims), start, seeds=4, phases=5, phase_steps=120, seed=7)
    prev = len(start)
    for lay, obj in zip(r["layouts"], r["objectives"]):
        check_valid(grid, dims, proto, lay)
        assert obj == len(lay) and obj <= prev
        prev = obj
    assert r["objectives"][-1] < len(start)
    assert r["steps_total"] > 0 and r["scored_total"] > 0


def test_model_weight_objective_non_increasing():
    grid = synth_terrain(40, 36, seed=5, t=2, density_q24=int(0.85 * (1 << 24)))
    dims, proto = keys_of(O.PLATFORMS_DEFAULT)
    costs = key_costs(dims, GUI_WEIGHTS)
    start = random_start(grid, dims, proto, seed=3)
    r = lns_placements_model(grid, dims, costs, start, seeds=4, phases=4, phase_steps=120, seed=1)
    prev = sum(costs[k] for _, _, k in start)
    for lay, obj in zip(r["layouts"], r["objectives"]):
        check_valid(grid, dims, proto, lay)
        assert obj == sum(costs[k] for _, _, k in lay) and obj <= prev
        prev = obj


def test_window_placements_constant_in_every_binding():
    with open(os.path.join(ROOT, "include", "tss.h")) as f:
        assert re.search(r"#define TSS_KERNEL_WINDOW_PLACEMENTS 5\b", f.read())
    with open(os.path.join(ROOT, "rust", "tss-sys", "src", "lib.rs")) as f:
        assert re.search(r"pub const TSS_KERNEL_WINDOW_PLACEMENTS: i32 = 5;", f.read())
    assert T.KERNEL_WINDOW_PLACEMENTS == 5
    from timberborn_support_solver_b200 import build as B
    assert "lns_placements.cu" in B.SOURCES


# ------------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def layout_keys(lay, dims):
    """PlatformLayout -> sorted [(x, y, key)] (keys by effective dims)"""
    out = []
    for p in lay.platforms().values():
        d = (p.definition.height, p.definition.width) if p.rotated else (p.definition.width, p.definition.height)
        out.append((p.x, p.y, dims.index(d)))
    return sorted(out)


BIT_EXACT = [((48, 40), 0.7), ((64, 64), 0.7), ((70, 33), 0.7), ((33, 90), 0.7), ((96, 72), 0.85)]


@pytest.mark.gpu
@pytest.mark.parametrize("seeds", [4, 8])
@pytest.mark.parametrize("shape,density", BIT_EXACT)
def test_window_placements_bit_exact_vs_model(eng, shape, density, seeds):
    w, h = shape
    grid = synth_terrain(w, h, seed=4, t=1, density_q24=int(density * (1 << 24)))
    run_bit_exact(eng, grid, O.PLATFORMS_DEFAULT, None, seeds)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["random-set", "gui-weights"])
def test_window_placements_bit_exact_vs_model_other_objectives(eng, case):
    if case == "random-set":
        run_bit_exact(eng, synth_terrain(50, 44, seed=3, t=1), RANDOM_SET, None, 4)
    else:
        run_bit_exact(eng, synth_terrain(60, 45, seed=5, t=2, density_q24=int(0.85 * (1 << 24))), O.PLATFORMS_DEFAULT, GUI_WEIGHTS, 4)


def run_bit_exact(eng, grid, defs, weights, seeds, phases=5, steps=150):
    dims, proto = keys_of(defs)
    costs = key_costs(dims, weights)
    s = eng.search(T.WorldGrid(grid), [T.PlatformDef(*d) for d in defs], seed=9, n_chains=seeds, chain_offset=30, kernel=T.KERNEL_WINDOW_PLACEMENTS)
    assert s.kernel_variant() == T.KERNEL_WINDOW_PLACEMENTS
    if weights:
        s.set_weights({T.PlatformDef(*d): v for d, v in weights.items()})
    start = layout_keys(s.best_layout(), dims)
    check_valid(grid, dims, proto, start)
    assert s.best_count() == sum(costs[k] for _, _, k in start)
    want = lns_placements_model(grid, dims, costs, start, seeds, phases, steps, seed=9, chain_offset=30)
    st0 = eng.stats()
    for p in range(phases):
        s.run(steps, -1)
        assert s.best_count() == want["objectives"][p], p
        assert layout_keys(s.best_layout(), dims) == want["layouts"][p], p
    st1 = eng.stats()
    assert st1["candidates_scored"] - st0["candidates_scored"] == want["scored_total"]
    assert st1["sls_steps"] - st0["sls_steps"] == want["steps_total"]
    assert want["objectives"][-1] < sum(costs[k] for _, _, k in start)   # the replay covered improvements, not just a fixed point
    s.close()


@pytest.mark.gpu
def test_window_placements_valid_at_scale(eng):
    grid = synth_terrain(256, 256, seed=1, t=0)                          # SURVEY.md C4
    dims, proto = keys_of(O.PLATFORMS_DEFAULT)
    layouts = []
    for _ in range(2):
        s = eng.search(T.WorldGrid(grid), T.PLATFORMS_DEFAULT, seed=3, kernel=T.KERNEL_WINDOW_PLACEMENTS)
        prev = s.best_count()
        start = prev
        for _ in range(8):
            s.run(2000, -1)
            lay = s.best_layout()
            plats = list(lay.platforms().values())
            assert O.validate(grid, [(p.x, p.y, p.definition.width, p.definition.height, int(p.rotated)) for p in plats]).is_valid
            assert all(p.definition in T.PLATFORMS_DEFAULT for p in plats)
            c = s.best_count()
            assert c == len(plats) and c <= prev
            prev = c
        assert prev < start
        layouts.append(layout_keys(lay, dims))
        s.close()
    assert layouts[0] == layouts[1]


@pytest.mark.gpu
def test_window_placements_never_worse_than_auto(eng):
    """The dense terrain of test_large_grid_with_larger_platforms_merges_supports, same seed and step budget."""
    grid = synth_terrain(96, 72, seed=4, t=1, density_q24=int(0.85 * (1 << 24)))
    counts = {}
    for name, kernel in (("auto", T.KERNEL_AUTO), ("window-placements", T.KERNEL_WINDOW_PLACEMENTS)):
        s = eng.search(T.WorldGrid(grid), T.PLATFORMS_DEFAULT, seed=5, kernel=kernel)
        for _ in range(4):
            s.run(1500, 0)
        counts[name] = s.best_layout().platform_count()
        s.close()
    assert counts["window-placements"] <= counts["auto"], counts


@pytest.mark.gpu
def test_window_placements_interface(eng):
    with pytest.raises(T.TssError):                                      # 32x32 and smaller: the placement search itself
        eng.search(T.WorldGrid(np.ones((32, 32), np.uint8)), T.PLATFORMS_DEFAULT, kernel=T.KERNEL_WINDOW_PLACEMENTS)
    big = T.WorldGrid(synth_terrain(48, 40, seed=1, t=5))
    with pytest.raises(T.TssError):                                      # {1x1} only: the 1x1 window decomposition
        eng.search(big, T.PLATFORMS_DEFAULT[:1], kernel=T.KERNEL_WINDOW_PLACEMENTS)
    with pytest.raises(T.TssError):                                      # a 7-long platform
        eng.search(big, [T.PlatformDef(1, 1), T.PlatformDef(1, 7)], kernel=T.KERNEL_WINDOW_PLACEMENTS)
    s = eng.search(big, T.PLATFORMS_DEFAULT, n_chains=5, kernel=T.KERNEL_WINDOW_PLACEMENTS)
    assert s.kernel_variant() == T.KERNEL_WINDOW_PLACEMENTS
    assert s.n_chains == 3 * 3 * 8                                       # windows at the widest offset x chains per window (5 -> 8)
    with pytest.raises(T.TssError):
        s.read_chains()
    with pytest.raises(T.TssError):
        s.read_placements()
    with pytest.raises(T.TssError):
        s.write_chains(np.zeros((s.n_chains, 32), np.uint32))
    st0 = eng.stats()
    c0 = s.best_count()
    s.run(300)
    s.best_count()                                                       # synchronises: the counters are folded in then
    st1 = eng.stats()
    for key in ("candidates_scored", "sls_steps", "sls_flips"):
        assert st1[key] > st0[key], key
    assert s.global_best() == s.best_count() <= c0
    s.set_bound(s.best_count())                                          # a bound from outside hides counts that do not beat it
    assert s.best_count() is None
    s.close()
    auto = eng.search(big, T.PLATFORMS_DEFAULT)                          # AUTO keeps the 1x1 window decomposition
    assert auto.kernel_variant() == 0
    auto.close()
