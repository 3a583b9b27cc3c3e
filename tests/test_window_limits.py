"""Per-type platform limits on grids larger than 32x32: the window placement search with per-window class budgets
(tss_search_create_with_limits, csrc/lns_placements.cu driving sls_multi_kernel<false, true, true>).

CPU: the scalar replay (tests/window_limits_model.py) keeps every layout valid and within every limit after every phase, its
budgets split exactly the slack, and without a binding budget it is the unlimited replay.
GPU: the device start layout is the trim of the unlimited start, the device follows the replay bit for bit, tss_solve_with_limits
and tss_solve_instance answer such instances, and the `-l` loops of solver_loop and tss_repl run on the GPU."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import synth_terrain
from test_window_placements import BIT_EXACT, GUI_WEIGHTS, check_valid, key_costs, keys_of, layout_keys, random_start
from window_limits_model import class_counts, limit_start, lns_placements_limits_model
from window_model import lns_placements_model

P = T.PlatformDef
LIMIT_SETS = {"5:2": {(5, 5): 2}, "3:1,5:1": {(3, 3): 1, (5, 5): 1}, "1x2:3": {(1, 2): 3}, "5:0": {(5, 5): 0}}
SHAPES = [(48, 40), (70, 33), (33, 90)]


def classes(defs, limits):
    keys, mask, lim = T.card_limit_classes([P(*d) for d in defs], {P(*d): v for d, v in limits.items()})
    assert keys == keys_of(defs)[0]
    return mask, lim


# ------------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("objective", ["count", "gui-weights"])
@pytest.mark.parametrize("name", list(LIMIT_SETS))
@pytest.mark.parametrize("shape", SHAPES)
def test_model_keeps_every_limit(shape, name, objective):
    w, h = shape
    grid = synth_terrain(w, h, seed=2, t=w + h)
    defs = [(d.width, d.height) for d in T.PLATFORMS_DEFAULT]
    dims, proto = keys_of(defs)
    mask, lim = classes(defs, LIMIT_SETS[name])
    costs = key_costs(dims, GUI_WEIGHTS if objective == "gui-weights" else None)
    start = limit_start(grid, dims, random_start(grid, dims, proto, seed=w * h), mask, lim)
    check_valid(grid, dims, proto, start)
    assert all(n <= l for n, l in zip(class_counts(start, mask, len(lim)), lim))
    r = lns_placements_limits_model(grid, dims, costs, start, seeds=4, phases=5, phase_steps=120, key_mask=mask, class_limit=lim, seed=7)
    prev = sum(costs[k] for _, _, k in start)
    for lay, obj, b, frozen, counts in zip(r["layouts"], r["objectives"], r["budgets"], r["frozen"], r["counts"]):
        check_valid(grid, dims, proto, lay)
        assert obj == sum(costs[k] for _, _, k in lay) and obj <= prev
        prev = obj
        assert counts == class_counts(lay, mask, len(lim)) and all(n <= l for n, l in zip(counts, lim))
        assert list(b.sum(axis=0)) == [l - f for l, f in zip(lim, frozen)]   # the budgets hand out exactly the slack
        assert (b >= 0).all()
    assert r["objectives"][-1] < sum(costs[k] for _, _, k in start)
    if not any(r["binding"]):                                            # no class was ever full: the unlimited replay
        want = lns_placements_model(grid, dims, costs, start, seeds=4, phases=5, phase_steps=120, seed=7)
        assert r["layouts"] == want["layouts"] and r["scored_total"] == want["scored_total"] and r["steps_total"] == want["steps_total"]


@pytest.mark.parametrize("limits,binds", [({(5, 5): 1000}, False), ({(3, 3): 1, (5, 5): 1}, True)], ids=["generous", "tight"])
def test_model_is_the_unlimited_replay_unless_a_budget_binds(limits, binds):
    grid = synth_terrain(48, 40, seed=2, t=88)
    defs = [(d.width, d.height) for d in T.PLATFORMS_DEFAULT]
    dims, proto = keys_of(defs)
    mask, lim = classes(defs, limits)
    start = limit_start(grid, dims, random_start(grid, dims, proto, seed=48 * 40), mask, lim)
    r = lns_placements_limits_model(grid, dims, [1] * len(dims), start, 4, 5, 120, mask, lim, seed=7)
    want = lns_placements_model(grid, dims, [1] * len(dims), start, 4, 5, 120, seed=7)
    assert any(r["binding"]) == binds
    assert (r["layouts"] == want["layouts"]) == (not binds)


def test_limit_start_trims_in_anchor_order():
    grid = synth_terrain(40, 36, seed=1, t=3)
    defs = [(d.width, d.height) for d in T.PLATFORMS_DEFAULT]
    dims, proto = keys_of(defs)
    start = random_start(grid, dims, proto, seed=5)
    mask, lim = classes(defs, {(1, 2): 2})
    out = limit_start(grid, dims, start, mask, lim)
    check_valid(grid, dims, proto, out)
    big = sorted((p for p in start if mask[p[2]]), key=lambda p: (p[1], p[0]))
    assert [p for p in out if mask[p[2]]] == sorted(big[:2])                # the first two of the class, row-major
    assert set(p for p in start if not mask[p[2]]) <= set(out)              # nothing outside a class is dropped
    assert all(dims[k] == (1, 1) for p in set(out) - set(start) for k in [p[2]])


def test_window_limits_in_every_binding():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "rust", "tss-sys", "src", "lib.rs")) as f:
        src = f.read()
    assert "pub fn tss_search_create_with_limits(" in src and "pub fn tss_engine_window_limits(" in src
    from timberborn_support_solver_b200 import _lib
    assert "tss_search_create_with_limits" in _lib.SIGNATURES and "tss_engine_window_limits" in _lib.SIGNATURES


# ------------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def run_limited_bit_exact(eng, grid, defs, limits, weights, seeds, phases=5, steps=150):
    dims, proto = keys_of(defs)
    mask, lim = classes(defs, limits)
    costs = key_costs(dims, weights)
    unl = eng.search(T.WorldGrid(grid), [P(*d) for d in defs], seed=9, n_chains=seeds, chain_offset=30, kernel=T.KERNEL_WINDOW_PLACEMENTS)
    greedy = layout_keys(unl.best_layout(), dims)
    unl.close()
    s = eng.search(T.WorldGrid(grid), [P(*d) for d in defs], seed=9, n_chains=seeds, chain_offset=30, limits={P(*d): v for d, v in limits.items()})
    assert s.kernel_variant() == T.KERNEL_WINDOW_PLACEMENTS
    if weights:
        s.set_weights({P(*d): v for d, v in weights.items()})
    start = layout_keys(s.best_layout(), dims)
    assert start == limit_start(grid, dims, greedy, mask, lim)          # the device trims the greedy cover as the replay does
    assert s.best_count() == sum(costs[k] for _, _, k in start)
    want = lns_placements_limits_model(grid, dims, costs, start, seeds, phases, steps, mask, lim, seed=9, chain_offset=30)
    st0 = eng.stats()
    for p in range(phases):
        s.run(steps, -1)
        assert s.best_count() == want["objectives"][p], p
        assert layout_keys(s.best_layout(), dims) == want["layouts"][p], p
    st1 = eng.stats()
    assert st1["candidates_scored"] - st0["candidates_scored"] == want["scored_total"]
    assert st1["sls_steps"] - st0["sls_steps"] == want["steps_total"]
    s.close()
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("seeds", [4, 8])
@pytest.mark.parametrize("shape,density", BIT_EXACT)
def test_window_limits_bit_exact_vs_model(eng, shape, density, seeds):
    w, h = shape
    grid = synth_terrain(w, h, seed=4, t=1, density_q24=int(density * (1 << 24)))
    want = run_limited_bit_exact(eng, grid, [(d.width, d.height) for d in T.PLATFORMS_DEFAULT], {(3, 3): 1, (5, 5): 1}, None, seeds)
    assert any(want["binding"])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["non-binding", "gui-weights", "terrain64-16keys"])
def test_window_limits_bit_exact_vs_model_other_cases(eng, case):
    defs8 = [(d.width, d.height) for d in T.PLATFORMS_DEFAULT]
    if case == "non-binding":
        grid = synth_terrain(48, 40, seed=4, t=1, density_q24=int(0.7 * (1 << 24)))
        want = run_limited_bit_exact(eng, grid, defs8, {(5, 5): 1000}, None, 4)
        assert not any(want["binding"])
        # with limits that never bind the device layouts are those of the unlimited search
        s = eng.search(T.WorldGrid(grid), T.PLATFORMS_DEFAULT, seed=9, n_chains=4, chain_offset=30, kernel=T.KERNEL_WINDOW_PLACEMENTS)
        dims = keys_of(defs8)[0]
        for p in range(5):
            s.run(150, -1)
            assert layout_keys(s.best_layout(), dims) == want["layouts"][p], p
        s.close()
    elif case == "gui-weights":
        grid = synth_terrain(60, 45, seed=5, t=2, density_q24=int(0.85 * (1 << 24)))
        run_limited_bit_exact(eng, grid, defs8, {(1, 2): 6, (5, 5): 1}, GUI_WEIGHTS, 4)
    else:
        keys16 = [(1, 1), (2, 2), (1, 2), (1, 3), (1, 5), (2, 3), (2, 5), (3, 4), (4, 6)]
        want = run_limited_bit_exact(eng, synth_terrain(64, 64, seed=4, t=2), keys16, {(2, 2): 4, (1, 5): 3, (3, 4): 1}, None, 4)
        assert any(want["binding"])


def plats_of(layout):
    return [(p.x, p.y, p.definition.width, p.definition.height, int(p.rotated)) for p in layout.platforms().values()]


def within(layout, limits):
    """class counts of a layout as the encoder counts them (a platform counts towards d if it contains d or d^T)"""
    for (dw, dh), v in limits.items():
        n = sum(1 for p in layout.platforms().values()
                if (dw <= p.definition.width and dh <= p.definition.height) or (dh <= p.definition.width and dw <= p.definition.height))
        if n > v:
            return False
    return True


@pytest.mark.gpu
@pytest.mark.parametrize("shape,density", [((48, 48), 0.7), ((96, 72), 0.85)])
@pytest.mark.parametrize("variant", ["per-type", "with-count", "weights"])
def test_solve_with_limits_on_large_grids(eng, shape, density, variant):
    w, h = shape
    grid = synth_terrain(w, h, seed=2, t=1, density_q24=int(density * (1 << 24)))
    g = T.WorldGrid(grid)
    per_type = {(5, 5): 2, (3, 3): 3}
    card = {P(*d): v for d, v in per_type.items()}
    if variant == "with-count":
        res, lay0, _ = eng.solve_with_limits(g, T.PLATFORMS_DEFAULT, T.PlatformLimits(dict(card)), seed=1, max_steps=2000)
        assert res == T.SAT
        card[P(1, 1)] = lay0.platform_count()
    lim = T.PlatformLimits(card, {P(*d): v for d, v in GUI_WEIGHTS.items()} if variant == "weights" else {}, None)
    res, layout, obj = eng.solve_with_limits(g, T.PLATFORMS_DEFAULT, lim, seed=1, max_steps=2000)
    assert res == T.SAT
    assert O.validate(grid, plats_of(layout)).is_valid and within(layout, per_type)
    if variant == "with-count":
        assert layout.platform_count() <= card[P(1, 1)]
    if variant != "weights":
        assert obj == layout.platform_count()
    with pytest.raises(T.TssError) as err:                               # a 1x7 def: no window placement search
        eng.solve_with_limits(g, [P(1, 1), P(1, 7), P(3, 3)], T.PlatformLimits({P(3, 3): 2}), seed=1, max_steps=500)
    assert err.value.code == T._lib.TSS_E_UNSUPPORTED


@pytest.mark.gpu
def test_create_with_limits_interface(eng):
    big = T.WorldGrid(synth_terrain(48, 40, seed=1, t=5))
    for bad in ({P(1, 1): 3}, {P(3, 3): -1}):
        with pytest.raises(T.TssError) as err:
            eng.search(big, T.PLATFORMS_DEFAULT, limits=bad)
        assert err.value.code == T._lib.TSS_E_INVALID
    with pytest.raises(T.TssError) as err:                               # another kernel
        eng.search(big, T.PLATFORMS_DEFAULT, limits={P(5, 5): 1}, kernel=T.KERNEL_WARP)
    assert err.value.code == T._lib.TSS_E_UNSUPPORTED
    s = eng.search(big, T.PLATFORMS_DEFAULT, limits={P(7, 7): 1})          # vacuous: the plain search (AUTO: the 1x1 decomposition)
    assert s.kernel_variant() == 0
    s.close()
    s = eng.search(big, T.PLATFORMS_DEFAULT, limits={P(5, 5): 1})
    assert s.kernel_variant() == T.KERNEL_WINDOW_PLACEMENTS
    with pytest.raises(T.TssError) as err:                               # set_card_limits keeps its contract on window searches
        s.set_card_limits({P(5, 5): 1})
    assert err.value.code == T._lib.TSS_E_UNSUPPORTED
    s.close()
    small = T.WorldGrid(synth_terrain(20, 17, seed=3, t=1))                 # up to 32x32: create + set_card_limits
    s = eng.search(small, T.PLATFORMS_DEFAULT, seed=1, n_chains=8, limits={P(5, 5): 0})
    s.run(200, 0)
    assert not any(p.definition == P(5, 5) for p in s.best_layout().platforms().values())
    s.close()


def _instance(eng, grid, limits):
    from timberborn_support_solver_b200 import _lib
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, T.WorldGrid(grid))
    cnf = enc.with_limits(T.PlatformLimits({P(*d): v for d, v in limits.items()}))
    dev = eng.upload_cnf(cnf)
    lits, offs = np.ascontiguousarray(cnf.lits, np.int32), np.ascontiguousarray(cnf.offsets, np.uint32)
    h, info = C.c_void_p(), _lib.InstanceInfo()
    assert eng.lib.tss_instance_find(lits.ctypes.data_as(C.POINTER(C.c_int32)), offs.ctypes.data_as(C.POINTER(C.c_uint32)), cnf.n_clauses, cnf.n_vars,
                                     C.byref(h), C.byref(info), None, 0) == _lib.TSS_SAT
    a = np.full(cnf.n_vars + 1, 2, np.uint8)
    rc = eng.lib.tss_solve_instance(eng._h, dev._h, h, C.byref(info), None, 1, 0, a.ctypes.data_as(C.POINTER(C.c_uint8)))
    eng.lib.tss_encoding_destroy(h)
    return rc, a


@pytest.mark.gpu
def test_solve_instance_with_window_limits(eng):
    from timberborn_support_solver_b200 import _lib
    grid = synth_terrain(48, 48, seed=2, t=1)                            # the instance test_type_limits.py leaves to the exact solver
    try:
        eng.window_limits(True)
        rc, a = _instance(eng, grid, {(5, 5): 3})
        assert rc == _lib.TSS_SAT
        assert O.Encoding(O.PLATFORMS_DEFAULT, grid).with_limits(card_limits={(5, 5): 3}).count_falsified(a)[0] == 0
        rc, _ = _instance(eng, grid, {(5, 5): 3, (1, 1): 1})               # an impossible count: unknown, never unsat
        assert rc == _lib.TSS_UNKNOWN
    finally:
        eng.window_limits(False)
    rc, _ = _instance(eng, grid, {(5, 5): 3})                             # off (the default): the exact solver's instance
    assert rc == _lib.TSS_UNKNOWN


@pytest.mark.gpu
def test_solver_loop_with_window_limits(eng):
    grid = synth_terrain(40, 36, seed=3, t=1)
    g = T.WorldGrid(grid)
    project = T.Project(T.World(g))
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, g)
    seen = []
    out = T.solver_loop(project, enc, T.PlatformLimits({P(5, 5): 1}), eng, exact_solver=None, seed=2, window_limits=True,
                        on_solution=lambda lay: seen.append(lay))
    gpu = [s for s in out["steps"] if s["result"] == T.SAT]
    assert len(gpu) >= 2 and all(s["source"] == "gpu" and s["valid"] for s in gpu)
    counts = [s["count"] for s in gpu]
    assert all(b < a for a, b in zip(counts, counts[1:]))
    assert all(within(lay, {(5, 5): 1}) for lay in seen)
    assert out["steps"][-1]["result"] == T.INTERRUPTED and not out["proved_optimal"]


@pytest.mark.gpu
def test_repl_window_limits(tmp_path):
    grid = synth_terrain(48, 48, seed=2, t=1)
    proj = tmp_path / "project.toml"
    proj.write_text(T.WorldGrid(grid).to_toml())
    exe = os.path.join(os.path.dirname(T.__file__), "tss_repl")
    out = subprocess.run([exe, str(proj), "--window-limits", "-l", "5:2", "--seed", "3"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    summary = [ln for ln in out.stdout.splitlines() if ln.startswith("# best=")][-1]
    assert 'verdict="unknown (no exact solver answer)"' in summary, out.stdout
    assert int(re.search(r"gpu_solves=(\d+)", summary).group(1)) >= 2, out.stdout
    assert "FAILED" not in out.stdout
