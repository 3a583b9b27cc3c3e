"""The placement search (sls_multi_kernel, platform sets beyond {1x1}) at the edges of what it takes: 32 columns and 32 rows,
one-row and one-column grids, keys that fit nowhere, a full set of 16 keys, 6x6 footprints against the right and bottom edge,
item lists far beyond one chunk of 32, steps beyond 32 768, and objectives whose costs differ.

CPU: the three scalar models rank additions by gain per cost — doubling every cost changes nothing but the objective — and
count flips (platforms added + removed) consistently with the list they keep.
GPU: the epoch kernel, LIMITS, WINDOW and the fused one-shot launch bit for bit against those models, flip counter included."""
import numpy as np
import pytest

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import golden, rows_to_grid, synth_terrain
from limits_model import limits_model
from test_window_placements import check_valid, key_costs, keys_of, layout_keys, random_start
from window_model import lns_placements_model

P = T.PlatformDef
NB = 1 << 20                                   # no bound (sls::NO_BOUND)
DEFAULT8 = [(d.width, d.height) for d in T.PLATFORMS_DEFAULT]
SQUARES = [(1, 1), (2, 2), (3, 3), (5, 5), (6, 6)]
KEYS16 = [(1, 1), (2, 2), (1, 2), (1, 3), (1, 5), (2, 3), (2, 5), (3, 4), (4, 6)]   # 1x1, 2x2 and 7 non-square defs: 16 keys
EPOCHS = [(40, NB, 0), (150, NB, 0), (400, NB, 0)]


def checkerboard(w, h):
    return ((np.arange(w)[None, :] + np.arange(h)[:, None]) % 2 == 0).astype(np.uint8)


def lattice(w, h):
    g = np.zeros((h, w), np.uint8)
    g[::2, ::2] = 1
    return g


def edge_terrain():
    """32x32 at density 0.7 with a solid band along the right and bottom edge, where 6x6 footprints end at x = 31 / y = 31"""
    g = synth_terrain(32, 32, seed=11, t=4)
    g[:, 26:] = 1
    g[26:, :] = 1
    return g


def fixture(name):
    return rows_to_grid(golden("fixtures")[name]["grid"])


def platforms_of(codes, dims, proto):
    return [(int(c) & 31, (int(c) >> 5) & 31, *proto[int(c) >> 10]) for c in codes]


def class_counts(codes, mask, n_classes):
    return [sum((mask[int(c) >> 10] >> j) & 1 for c in codes) for j in range(n_classes)]


# ------------------------------------------------------------------------------------------------------------------ CPU
DOUBLING = {   # (defs, costs per key in keys_of order): powers of two keep 64 / cost exact, so halving the rank is exact too
    "1-2-4": ([(1, 1), (1, 2), (3, 3)], [1, 2, 2, 4]),
    "1-2-4-16-32": ([(1, 1), (1, 2), (2, 2), (3, 3), (4, 4)], [1, 2, 2, 4, 16, 32]),
}


def _run_model(model, grid, dims, costs, n_chains=6, epochs=EPOCHS):
    if model == "slsm":
        return O.slsm_model(grid, dims, costs, n_chains, epochs, seed=9, chain_offset=50, count_flips=True)
    if model == "limits":    # one class that never fills (3x3 and larger at most 100): the LIMITS step rule with its class counters
        mask = [int(w >= 3 and h >= 3) for w, h in dims]
        return limits_model(grid, dims, costs, mask, [100], n_chains, epochs, seed=9, chain_offset=50, count_flips=True)
    raise AssertionError(model)


@pytest.mark.parametrize("case", list(DOUBLING))
@pytest.mark.parametrize("model", ["slsm", "limits"])
def test_cost_doubling_is_invisible(model, case):
    """Additions are ranked by gain per cost: doubling every cost doubles the objective and changes nothing else.  (A rank that
    scales only the cost-1 key — g for cost 1, 64 g / cost otherwise — ranks that key 64 times too low, and the two runs part.)"""
    defs, costs = DOUBLING[case]
    dims, _ = keys_of(defs)
    assert len(dims) == len(costs)
    grid = synth_terrain(20, 17, seed=3, t=1)
    a = _run_model(model, grid, dims, costs)
    b = _run_model(model, grid, dims, [2 * c for c in costs])
    for key in ("items", "k", "best_items", "best_k", "step"):
        assert np.array_equal(a[key], b[key]), key
    assert np.array_equal(np.where(a["best"] < NB, 2 * a["best"], NB), b["best"])
    for key in ("scored_total", "steps_total", "flips_total"):
        assert a[key] == b[key], key
    assert (a["best"] < NB).any() and a["k"].any()


@pytest.mark.parametrize("case", list(DOUBLING))
def test_cost_doubling_is_invisible_in_the_window_model(case):
    defs, costs = DOUBLING[case]
    dims, proto = keys_of(defs)
    grid = synth_terrain(48, 40, seed=2, t=3)
    start = random_start(grid, dims, proto, seed=5)                     # built on the host: random platforms, 1x1 where still needed
    a = lns_placements_model(grid, dims, costs, start, seeds=4, phases=2, phase_steps=120, seed=7, chain_offset=5)
    b = lns_placements_model(grid, dims, [2 * c for c in costs], start, seeds=4, phases=2, phase_steps=120, seed=7, chain_offset=5)
    assert a["layouts"] == b["layouts"]
    assert [2 * o for o in a["objectives"]] == b["objectives"]
    for key in ("scored_total", "steps_total", "flips_total"):
        assert a[key] == b[key], key
    assert a["objectives"][-1] < sum(costs[k] for _, _, k in start)
    check_valid(grid, dims, proto, a["layouts"][-1])


@pytest.mark.parametrize("model", ["slsm", "limits"])
def test_flip_bookkeeping_step_by_step(model):
    """One chain, runs of 0 .. 160 steps (one epoch each, so every run is a prefix of the next): a step flips 0, 1 or 2
    platforms, and adds - removes = the change of k — (0, 0), (1, +1), (1, -1) or (2, 0) per step."""
    grid = synth_terrain(14, 12, seed=5, t=2)
    dims, _ = keys_of(DEFAULT8)
    costs = [1] * len(dims)
    prev = None
    seen = set()
    for m in range(0, 161):
        r = _run_model(model, grid, dims, costs, n_chains=1, epochs=[(m, NB, 0)] if m else [])
        cur = (r["flips_total"], int(r["k"][0]), r["steps_total"])
        if prev is not None:
            df, dk, ds = cur[0] - prev[0], cur[1] - prev[1], cur[2] - prev[2]
            assert ds == 1 and (df, dk) in {(0, 0), (1, 1), (1, -1), (2, 0)}, (m, df, dk)
            seen.add((df, dk))
        prev = cur
    assert {(1, 1), (1, -1), (2, 0)} <= seen        # additions, drops and swaps all happened


def test_flip_totals_on_many_chains():
    grid = checkerboard(16, 12)
    dims, _ = keys_of([(1, 1), (1, 2)])
    r = O.slsm_model(grid, dims, [1] * len(dims), 5, [(150, NB, 0), (100, 90, 0)], seed=3, chain_offset=7, count_flips=True)
    adds2 = r["flips_total"] + int(r["k"].sum())                       # chains start empty: adds - removes = sum of k
    assert r["flips_total"] > 0 and adds2 % 2 == 0 and r["flips_total"] >= int(r["k"].sum())
    assert r["flips_total"] <= 2 * r["steps_total"]
    dims8, _ = keys_of(DEFAULT8)
    grid = synth_terrain(48, 40, seed=2, t=3)
    start = [(int(x), int(y), 0) for y, x in zip(*np.nonzero(grid))]
    w = lns_placements_model(grid, dims8, [1] * len(dims8), start, seeds=4, phases=2, phase_steps=100, seed=1)
    assert 0 < w["flips_total"] <= 2 * w["steps_total"]


# ------------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def _search(eng, grid, defs, weights=None, **kw):
    s = eng.search(T.WorldGrid(grid), [P(*d) for d in defs], **kw)
    if weights:
        s.set_weights({P(*d): v for d, v in weights.items()})
    return s


def _run_epochs(eng, s, epochs):
    st0 = eng.stats()
    for steps, bound, target in epochs:
        if bound < NB:
            s.set_bound(bound)
        s.run(steps, target)
    got = s.read_placements()
    st1 = eng.stats()
    return got, {k: st1[k] - st0[k] for k in ("candidates_scored", "sls_steps", "sls_flips")}


def _assert_same(got, delta, want):
    for key in ("k", "best", "best_k", "step"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(got["items"], want["items"]) and np.array_equal(got["best_items"], want["best_items"])
    assert delta == dict(candidates_scored=want["scored_total"], sls_steps=want["steps_total"], sls_flips=want["flips_total"])


PARITY = {   # name: (grid, defs, weights, n_chains, chain_offset, epochs)
    "rect32-default8": (lambda: np.ones((32, 32), np.uint8), DEFAULT8, None, 7, 50, EPOCHS),
    "edge32-squares": (edge_terrain, SQUARES, None, 7, 13, EPOCHS),
    "row32x1-default8": (lambda: np.ones((1, 32), np.uint8), DEFAULT8, None, 5, 3, [(30, NB, 0), (120, NB, 0)]),
    "col1x32-default8": (lambda: np.ones((32, 1), np.uint8), DEFAULT8, None, 9, 77, [(30, NB, 0), (120, NB, 0)]),
    "terrain31x29-16keys": (lambda: synth_terrain(31, 29, seed=8, t=5), KEYS16, None, 7, 21, EPOCHS),
    "4x4-keys-out-of-bounds": (lambda: np.ones((4, 4), np.uint8), [(1, 1), (1, 2), (5, 5), (6, 6)], None, 5, 1, [(60, NB, 0), (200, NB, 0)]),
    "density0.5-32": (lambda: synth_terrain(32, 32, seed=6, t=3, density_q24=1 << 23), DEFAULT8, None, 7, 40, EPOCHS),
    "checkerboard32": (lambda: checkerboard(32, 32), [(1, 1), (1, 2)], None, 5, 9, [(700, NB, 0), (150, NB, 0), (300, 511, 0)]),
    "lattice32": (lambda: lattice(32, 32), [(1, 1), (1, 2), (2, 2)], None, 7, 2, [(350, NB, 0), (200, NB, 0)]),
    "ex1-40000-steps": (lambda: fixture("ex1"), DEFAULT8, None, 5, 60, [(40000, NB, 0)]),
    "weights-1-1-2": (lambda: synth_terrain(20, 17, seed=3, t=1), [(1, 1), (1, 2), (2, 2)], {(1, 1): 1, (1, 2): 1, (2, 2): 2}, 7, 50, EPOCHS),
}


def _check_case(name, grid, dims, proto, want):
    """What each case is there for actually happened in the trajectories compared."""
    def codes():
        for c in range(len(want["k"])):
            yield from want["items"][c][: want["k"][c]]
            yield from want["best_items"][c][: want["best_k"][c]]
    if name == "rect32-default8":
        assert any((int(c) & 31) + dims[int(c) >> 10][0] == 32 for c in codes())            # a footprint on column 31
    if name == "edge32-squares":
        six = dims.index((6, 6))
        assert any(int(c) >> 10 == six and (int(c) & 31) == 26 for c in codes())
        assert any(int(c) >> 10 == six and ((int(c) >> 5) & 31) == 26 for c in codes())
    if name == "checkerboard32":
        assert want["best"].min() == 512 and want["k"].max() >= 480                        # 16 removal chunks
    if name == "lattice32":
        assert want["best"].min() == 256
    if name == "4x4-keys-out-of-bounds":
        assert not any(int(c) >> 10 >= dims.index((5, 5)) for c in codes())
    if name == "ex1-40000-steps":
        assert (want["step"] > 32768).all()
    for c in np.nonzero(want["best"] < NB)[0][:3]:
        assert O.validate(grid, platforms_of(want["best_items"][c][: want["best_k"][c]], dims, proto)).is_valid


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PARITY))
def test_placement_search_edges_bit_exact_vs_model(eng, name):
    make, defs, weights, n_chains, offset, epochs = PARITY[name]
    grid = make()
    s = _search(eng, grid, defs, weights, seed=9, n_chains=n_chains, chain_offset=offset)
    got, delta = _run_epochs(eng, s, epochs)
    s.close()
    dims, proto = keys_of(defs)
    assert got["key_dims"] == dims
    costs = key_costs(dims, weights)
    # (an epoch of the placement search is not split at 32 768 steps: its tabu marks are placement codes, not 16-bit stamps)
    want = O.slsm_model(grid, dims, costs, n_chains, epochs, seed=9, chain_offset=offset, count_flips=True)
    _assert_same(got, delta, want)
    assert (want["best"] < NB).any()
    _check_case(name, grid, dims, proto, want)


LIMITS = {   # name: (grid, defs, limits, n_chains, chain_offset, epochs)
    "rect32-3x3": (lambda: np.ones((32, 32), np.uint8), DEFAULT8, {(3, 3): 2}, 7, 50, EPOCHS),
    "checkerboard32-1x2": (lambda: checkerboard(32, 32), [(1, 1), (1, 2)], {(1, 2): 300}, 5, 9, [(700, NB, 0), (300, 511, 0)]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LIMITS))
def test_limited_search_edges_bit_exact_vs_model(eng, name):
    make, defs, limits, n_chains, offset, epochs = LIMITS[name]
    grid = make()
    s = _search(eng, grid, defs, seed=9, n_chains=n_chains, chain_offset=offset)
    s.set_card_limits({P(*d): v for d, v in limits.items()})
    got, delta = _run_epochs(eng, s, epochs)
    s.close()
    keys, mask, lim = T.card_limit_classes([P(*d) for d in defs], {P(*d): v for d, v in limits.items()})
    assert keys == got["key_dims"] and lim
    want = limits_model(grid, keys, [1] * len(keys), mask, lim, n_chains, epochs, seed=9, chain_offset=offset,
                        count_flips=True)
    _assert_same(got, delta, want)
    assert (want["best"] < NB).any()
    for c in range(n_chains):
        for items, k in ((got["items"][c], got["k"][c]), (got["best_items"][c], got["best_k"][c])):
            assert all(n <= L for n, L in zip(class_counts(items[:k], mask, len(lim)), lim)), (c, limits)
    if name == "checkerboard32-1x2":
        assert want["k"].min() > 32 and want["best"].min() == 512


WINDOWS = {   # name: (grid, defs, seeds, phases, steps)
    "checkerboard48x40": (lambda: checkerboard(48, 40), [(1, 1), (1, 2)], 4, 3, 150),
    "terrain64-16keys": (lambda: synth_terrain(64, 64, seed=4, t=2), KEYS16, 4, 4, 150),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WINDOWS))
def test_window_placements_edges_bit_exact_vs_model(eng, name):
    make, defs, seeds, phases, steps = WINDOWS[name]
    grid = make()
    dims, proto = keys_of(defs)
    s = _search(eng, grid, defs, seed=9, n_chains=seeds, chain_offset=30, kernel=T.KERNEL_WINDOW_PLACEMENTS)
    assert s.kernel_variant() == T.KERNEL_WINDOW_PLACEMENTS
    start = layout_keys(s.best_layout(), dims)
    check_valid(grid, dims, proto, start)
    want = lns_placements_model(grid, dims, [1] * len(dims), start, seeds, phases, steps, seed=9, chain_offset=30)
    st0 = eng.stats()
    for p in range(phases):
        s.run(steps, -1)
        assert s.best_count() == want["objectives"][p], p
        assert layout_keys(s.best_layout(), dims) == want["layouts"][p], p
    st1 = eng.stats()
    s.close()
    assert st1["candidates_scored"] - st0["candidates_scored"] == want["scored_total"]
    assert st1["sls_steps"] - st0["sls_steps"] == want["steps_total"]
    assert st1["sls_flips"] - st0["sls_flips"] == want["flips_total"]
    if name == "checkerboard48x40":
        assert want["objectives"][-1] == int(grid.sum())                # every platform holds exactly one ceiling tile


FUSED = {   # name: (grid, defs, card_limit)
    "rect32-default8": (lambda: np.ones((32, 32), np.uint8), DEFAULT8, None),
    "row32x1-default8": (lambda: np.ones((1, 32), np.uint8), DEFAULT8, 11),
    "checkerboard32": (lambda: checkerboard(32, 32), [(1, 1), (1, 2)], None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FUSED))
def test_fused_one_shot_launch_at_the_edges(name):
    """The second solve_upper_bound on the same platform set runs its first epoch as one fused launch: same layout as the
    first (epoch by epoch) call, fewer launches, and the layout passes the reference's validate()."""
    make, defs, limit = FUSED[name]
    grid = make()
    g = T.WorldGrid(grid)
    e = T.Engine(0)
    try:
        res_a, lay_a = e.solve_upper_bound(g, [P(*d) for d in defs], card_limit=limit, seed=4)
        launches_a = e.stats()["kernel_launches"]
        res_b, lay_b = e.solve_upper_bound(g, [P(*d) for d in defs], card_limit=limit, seed=4)
        launches_b = e.stats()["kernel_launches"] - launches_a
    finally:
        e.close()
    assert res_a == res_b == T.SAT and launches_b < launches_a
    tup = lambda p: (p.x, p.y, p.definition.width, p.definition.height, int(p.rotated))
    pa, pb = sorted(tup(p) for p in lay_a.platforms().values()), sorted(tup(p) for p in lay_b.platforms().values())
    assert pa == pb and O.validate(grid, pb).is_valid
    if limit is not None:
        assert len(pb) <= limit


@pytest.mark.gpu
def test_cost_doubling_is_invisible_on_the_device(eng):
    defs = [(1, 1), (1, 2), (2, 2)]
    grid = synth_terrain(24, 20, seed=7, t=2)
    runs = []
    for weights in ({(1, 1): 1, (1, 2): 1, (2, 2): 2}, {(1, 1): 2, (1, 2): 2, (2, 2): 4}):
        s = _search(eng, grid, defs, weights, seed=5, n_chains=7, chain_offset=11)
        got, delta = _run_epochs(eng, s, EPOCHS)
        s.close()
        runs.append((got, delta))
    (a, da), (b, db) = runs
    for key in ("items", "k", "best_items", "best_k", "step"):
        assert np.array_equal(a[key], b[key]), key
    assert np.array_equal(np.where(a["best"] < NB, 2 * a["best"], NB), b["best"]) and (a["best"] < NB).any()
    assert da == db


def test_limits_model_without_classes_counts_the_oracle_flips():
    grid = synth_terrain(14, 12, seed=5, t=2)
    dims, _ = keys_of(DEFAULT8)
    epochs = [(60, NB, 0), (200, NB, 0)]
    got = limits_model(grid, dims, [1] * len(dims), [0] * len(dims), [], 5, epochs, seed=4, chain_offset=3, count_flips=True)
    want = O.slsm_model(grid, dims, [1] * len(dims), 5, epochs, seed=4, chain_offset=3, count_flips=True)
    assert set(got) == set(want)
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k
    assert want["flips_total"] > 0
