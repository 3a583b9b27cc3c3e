"""Per-type platform limits (`solve -l k:v`, PlatformLimits.card_limits beyond 1x1) steering the placement search.

CPU: the class rule (tss_card_limit_classes) against the oracle's own encoder, and the scalar model with limits.
GPU: the LIMITS kernel bit for bit against that model, the REPL's `-l` loops, the instance bridge, the error codes of
tss_search_set_card_limits and the workspace a one-shot solve leaves behind."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import golden, synth_terrain
from limits_model import limits_model

P = T.PlatformDef
ONE = P(1, 1)
RANDOM_SET = [P(1, 1), P(2, 3), P(2, 2), P(1, 4), P(4, 4)]
GUI_WEIGHTS = {P(1, 1): 5, P(1, 2): 1, P(1, 3): 1, P(1, 4): 1, P(1, 5): 1, P(1, 6): 1, P(3, 3): 2, P(5, 5): 4}   # crates/gui/src/app.rs:53-62


def dims_le(a, b):
    return a[0] <= b[0] and a[1] <= b[1]


def class_counts(codes, mask, n_classes):
    return [sum((mask[c >> 10] >> j) & 1 for c in codes) for j in range(n_classes)]


# ------------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("defs", [[(d.width, d.height) for d in T.PLATFORMS_DEFAULT], [(d.width, d.height) for d in RANDOM_SET]],
                         ids=["default8", "random-set"])
def test_class_rule_matches_the_oracle_encoder(defs):
    """One platform of key q under with_limits({d: 0}) is a propagation conflict in the oracle's CNF exactly when q is in the
    class the engine derives for d: for every key q and every type d (keys, squares and rectangles outside the set)."""
    grid = np.ones((8, 8), np.uint8)
    enc = O.Encoding(defs, grid)
    types = sorted({(min(w, h), max(w, h)) for w, h in enc.dims} | {(2, 2), (4, 4), (6, 6), (2, 3), (2, 5), (3, 4), (1, 2), (3, 3)})
    for d in types:
        if d == (1, 1):
            continue
        cnf = enc.with_limits(card_limits={d: 0})
        keys, mask, lim = T.card_limit_classes([P(*x) for x in defs], {P(*d): 0})
        assert lim in ([], [0])
        for qi, q in enumerate(enc.dims):
            a = np.full(cnf.n_vars + 1, 2, np.uint8)
            a[enc.plat_var[0, qi]] = 1      # one platform of key q anchored at (0, 0): in bounds on 8x8
            _, conflict, _ = cnf.propagate(a)
            assert (conflict >= 0) == bool(mask[keys.index(q)]), (defs, d, q)


def test_class_rule_records():
    """1x1 records and vacuous ones make no class, a limit of 1024 or more is vacuous, equal classes merge into the smaller limit,
    a negative limit is an error."""
    keys, mask, lim = T.card_limit_classes(T.PLATFORMS_DEFAULT, {ONE: 3, P(2, 2): 1, P(5, 5): 1024, P(4, 6): 0})
    assert lim == [] and not any(mask)
    keys, mask, lim = T.card_limit_classes(T.PLATFORMS_DEFAULT, {P(1, 6): 4, P(6, 1): 2})
    assert lim == [2] and [keys[i] for i in range(len(keys)) if mask[i]] == [(1, 6), (6, 1)]
    keys, mask, lim = T.card_limit_classes(T.PLATFORMS_DEFAULT, {P(1, 2): 0})
    assert lim == [0] and [k for k, m in zip(keys, mask) if not m] == [(1, 1)]
    keys, mask, lim = T.card_limit_classes(T.PLATFORMS_DEFAULT[:1], {P(1, 2): 0, P(3, 3): 1})
    assert keys == [(1, 1)] and lim == []
    with pytest.raises(T.TssError):
        T.card_limit_classes(T.PLATFORMS_DEFAULT, {P(3, 3): -1})


def test_model_without_classes_is_the_oracle_model():
    grid = synth_terrain(14, 12, seed=5, t=2)
    keys, mask, lim = T.card_limit_classes(T.PLATFORMS_DEFAULT, {})
    epochs = [(60, 1 << 20, 0), (200, 1 << 20, 0)]
    got = limits_model(grid, keys, [1] * len(keys), mask, lim, 5, epochs, seed=4, chain_offset=3)
    want = O.slsm_model(grid, keys, [1] * len(keys), 5, epochs, seed=4, chain_offset=3)
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k


@pytest.mark.parametrize("case", range(6))
def test_model_keeps_every_limit(case):
    rng = np.random.default_rng(100 + case)
    w, h = int(rng.integers(8, 21)), int(rng.integers(8, 21))
    grid = (rng.random((h, w)) < 0.75).astype(np.uint8)
    defs = list(T.PLATFORMS_DEFAULT) if case % 2 == 0 else RANDOM_SET
    pool = [d for d in defs if d != ONE]
    limits = {pool[i]: int(rng.integers(0, 4)) for i in rng.choice(len(pool), size=2, replace=False)}
    keys, mask, lim = T.card_limit_classes(defs, limits)
    assert lim
    costs = [1] * len(keys) if case < 3 else [int(c) for c in rng.integers(1, 5, len(keys))]
    got = limits_model(grid, keys, costs, mask, lim, 8, [(150, 1 << 20, 0), (400, 1 << 20, 0)], seed=case)
    for c in range(8):
        for items, k in ((got["items"][c], got["k"][c]), (got["best_items"][c], got["best_k"][c])):
            assert all(n <= L for n, L in zip(class_counts(items[:k], mask, len(lim)), lim)), (case, c, limits)
    assert (got["best"] < (1 << 20)).any()


# ------------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def fixtures():
    from conftest import rows_to_grid
    return {k: rows_to_grid(v["grid"]) for k, v in golden("fixtures").items()}


PARITY = {
    "ex2-5x5": ("ex2", None, {P(5, 5): 2}, None),
    "ex1-3x3-1x4": ("ex1", None, {P(3, 3): 1, P(1, 4): 2}, None),
    "random-set": ("random", RANDOM_SET, {P(2, 2): 3, P(1, 4): 1}, None),
    "gui-weights": ("gui", None, {P(5, 5): 1, P(1, 3): 4}, GUI_WEIGHTS),
    "limit-0": ("ex3", None, {P(3, 3): 0, P(1, 5): 1}, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PARITY))
def test_limited_search_bit_exact_vs_model(eng, fixtures, case):
    name, defs, limits, weights = PARITY[case]
    defs = list(defs or T.PLATFORMS_DEFAULT)
    if name == "random":
        grid = synth_terrain(20, 17, seed=3, t=1)
    elif name == "gui":
        grid = synth_terrain(14, 12, seed=5, t=2, density_q24=int(0.85 * (1 << 24)))
    else:
        grid = fixtures[name]
    n_chains, offset, seed = 6, 50, 9
    epochs = [(40, 1 << 20, 0), (150, 1 << 20, 0), (400, 1 << 20, 0)]
    s = eng.search(T.WorldGrid(grid), defs, seed=seed, n_chains=n_chains, chain_offset=offset)
    if weights:
        s.set_weights(weights)
    s.set_card_limits(limits)
    st0 = eng.stats()
    for steps, _, target in epochs:
        s.run(steps, target)
    got = s.read_placements()
    st1 = eng.stats()
    keys, mask, lim = T.card_limit_classes(defs, limits)
    assert keys == got["key_dims"] and lim
    costs = [1] * len(keys)
    if weights:
        canon = lambda w, h: (min(w, h), max(w, h))
        costs = [sum(v for d, v in weights.items() if dims_le(canon(d.width, d.height), canon(w, h))) for w, h in keys]
    want = limits_model(grid, keys, costs, mask, lim, n_chains, epochs, seed=seed, chain_offset=offset)
    for key in ("k", "best", "best_k", "step"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(got["items"], want["items"]) and np.array_equal(got["best_items"], want["best_items"])
    assert st1["candidates_scored"] - st0["candidates_scored"] == want["scored_total"]
    assert st1["sls_steps"] - st0["sls_steps"] == want["steps_total"]
    for c in range(n_chains):
        for items, k in ((got["items"][c], got["k"][c]), (got["best_items"][c], got["best_k"][c])):
            assert all(n <= L for n, L in zip(class_counts(items[:k], mask, len(lim)), lim)), (c, limits)
    assert (want["best"] < (1 << 20)).any()
    if any(L == 0 for L in lim):
        blocked = [i for i, m in enumerate(mask) if any((m >> j) & 1 and lim[j] == 0 for j in range(len(lim)))]
        assert not any((code >> 10) in blocked for c in range(n_chains) for code in got["best_items"][c][: got["best_k"][c]])
    s.close()


def oracle_optimum(grid, defs, card):
    """The REPL's loop (crates/repl/src/main.rs:280-366) on the oracle with per-type limits: solve, count = platforms,
    1x1 limit = count - 1, until the CDCL stand-in says UNSAT.  -> proven minimum count."""
    enc = O.Encoding(defs, grid)
    best, limits = None, dict(card)
    while True:
        r, a, _ = enc.with_limits(card_limits=limits).solve()
        if r != 10:
            return best
        best = len(enc.layout_from_assignment(a))
        limits[(1, 1)] = best - 1


def _run_repl(tmp_path, grid, *args):
    proj = tmp_path / "project.toml"
    proj.write_text(T.WorldGrid(grid).to_toml())
    exe = os.path.join(os.path.dirname(T.__file__), "tss_repl")
    exact = f"{sys.executable} {os.path.join(os.path.dirname(__file__), 'exact_dimacs.py')}"
    out = subprocess.run([exe, str(proj), "--exact", exact, *args], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    summary = [ln for ln in out.stdout.splitlines() if ln.startswith("# best=")][-1]
    fields = dict(kv.split("=", 1) for kv in re.sub(r'verdict="[^"]*" ', "", summary[2:]).split(" ") if "=" in kv)
    counts = [int(ln.split("(")[1].split()[0]) for ln in out.stdout.splitlines() if ln.startswith("Solution found")]
    return out.stdout, fields, counts


REPL = [("ex1", "3:1,1x4:2", {(3, 3): 1, (1, 4): 2}), ("ex2", "5:2", {(5, 5): 2}), ("ex2", "5:1,1x6:2", {(5, 5): 1, (1, 6): 2}),
        ("ex3", "3:2,1x2:3", {(3, 3): 2, (1, 2): 3}), ("random", "5:1,3:2", {(5, 5): 1, (3, 3): 2})]


@pytest.mark.gpu
@pytest.mark.parametrize("name,arg,card", REPL, ids=[f"{n}:{a}" for n, a, _ in REPL])
def test_repl_limits_loop_reaches_the_optimum_on_the_gpu(eng, fixtures, tmp_path, name, arg, card):
    grid = synth_terrain(18, 16, seed=7, t=3) if name == "random" else fixtures[name]
    optimum = oracle_optimum(grid, O.PLATFORMS_DEFAULT, card)
    for extra in ((), ("--no-lower-bound",)):
        text, f, counts = _run_repl(tmp_path, grid, "-l", arg, "--seed", "3", *extra)
        assert int(f["best"]) == optimum and counts[-1] == optimum, (text, optimum)
        assert all(b < a for a, b in zip(counts, counts[1:]))
        assert text.count("Solution validation OK (gpu)") == len(counts) and "(exact)" not in text
        assert int(f["exact_solves"]) <= 1 and "FAILED" not in text


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ex1", "ex3"])
def test_limit_zero_reduces_the_platform_set(eng, fixtures, tmp_path, name):
    optimum = golden("proofs")[f"{name}/1x1"]["optimum"]
    text, f, counts = _run_repl(tmp_path, fixtures[name], "-l", "1x2:0", "--seed", "3")
    assert int(f["best"]) == optimum
    res, layout, obj = eng.solve_with_limits(T.WorldGrid(fixtures[name]), T.PLATFORMS_DEFAULT, T.PlatformLimits({P(1, 2): 0}), seed=1, max_steps=4000)
    assert res == T.SAT and all(p.definition == ONE for p in layout.platforms().values()) and obj == layout.platform_count()


@pytest.mark.gpu
def test_solve_instance_answers_limited_instances(eng, fixtures):
    from timberborn_support_solver_b200 import _lib
    lib = eng.lib
    grid = fixtures["ex2"]
    card = {(5, 5): 1, (1, 6): 2, (1, 1): 30}
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, T.WorldGrid(grid))
    cnf = enc.with_limits(T.PlatformLimits({P(*d): v for d, v in card.items()}))
    dev = eng.upload_cnf(cnf)
    lits, offs = np.ascontiguousarray(cnf.lits, np.int32), np.ascontiguousarray(cnf.offsets, np.uint32)
    info = _lib.InstanceInfo()
    h = C.c_void_p()
    assert lib.tss_instance_find(lits.ctypes.data_as(C.POINTER(C.c_int32)), offs.ctypes.data_as(C.POINTER(C.c_uint32)), cnf.n_clauses, cnf.n_vars,
                                 C.byref(h), C.byref(info), None, 0) == _lib.TSS_SAT
    a = np.full(cnf.n_vars + 1, 2, np.uint8)
    rc = lib.tss_solve_instance(eng._h, dev._h, h, C.byref(info), None, 1, 0, a.ctypes.data_as(C.POINTER(C.c_uint8)))
    assert rc == _lib.TSS_SAT
    o = O.Encoding(O.PLATFORMS_DEFAULT, grid).with_limits(card_limits=card)
    assert o.count_falsified(a)[0] == 0
    lib.tss_encoding_destroy(h)
    # a handle that carries no recorded limits (tss_encoding_create), with the same info: left to the exact solver
    a[:] = 2
    assert lib.tss_solve_instance(eng._h, dev._h, enc._h, C.byref(info), None, 1, 0, a.ctypes.data_as(C.POINTER(C.c_uint8))) == _lib.TSS_UNKNOWN
    # 48x48 with per-type limits: the window searches do not steer by them
    big = synth_terrain(48, 48, seed=2, t=1)
    enc2 = T.Encoding.encode(T.PLATFORMS_DEFAULT, T.WorldGrid(big))
    cnf2 = enc2.with_limits(T.PlatformLimits({P(5, 5): 3}))
    dev2 = eng.upload_cnf(cnf2)
    l2, o2 = np.ascontiguousarray(cnf2.lits, np.int32), np.ascontiguousarray(cnf2.offsets, np.uint32)
    h2, info2 = C.c_void_p(), _lib.InstanceInfo()
    assert lib.tss_instance_find(l2.ctypes.data_as(C.POINTER(C.c_int32)), o2.ctypes.data_as(C.POINTER(C.c_uint32)), cnf2.n_clauses, cnf2.n_vars,
                                 C.byref(h2), C.byref(info2), None, 0) == _lib.TSS_SAT
    a2 = np.full(cnf2.n_vars + 1, 2, np.uint8)
    assert lib.tss_solve_instance(eng._h, dev2._h, h2, C.byref(info2), None, 1, 0, a2.ctypes.data_as(C.POINTER(C.c_uint8))) == _lib.TSS_UNKNOWN
    lib.tss_encoding_destroy(h2)


@pytest.mark.gpu
def test_set_card_limits_error_codes(eng, fixtures):
    g = T.WorldGrid(fixtures["ex1"])
    s = eng.search(g, T.PLATFORMS_DEFAULT, seed=1, n_chains=8)
    for bad in ({ONE: 3}, {P(3, 3): -1}):
        with pytest.raises(T.TssError) as e:
            s.set_card_limits(bad)
        assert e.value.code == -1
    s.set_card_limits({P(2, 2): 1, P(5, 5): 2000})     # vacuous: accepted, no class
    s.run(10)
    with pytest.raises(T.TssError) as e:
        s.set_card_limits({P(3, 3): 1})
    assert e.value.code == -1                          # after the first run
    s.close()
    s = eng.search(g, T.PLATFORMS_DEFAULT[:1], seed=1)
    s.set_card_limits({P(3, 3): 0, P(1, 2): 1})        # {1x1}-only: every record is vacuous
    s.close()
    big = T.WorldGrid(synth_terrain(48, 48, seed=2, t=1))
    for kernel in (0, T.KERNEL_WINDOW_PLACEMENTS):
        s = eng.search(big, T.PLATFORMS_DEFAULT, seed=1, kernel=kernel)
        s.set_card_limits({P(2, 2): 1})                # vacuous: fine on windows too
        with pytest.raises(T.TssError) as e:
            s.set_card_limits({P(5, 5): 2})
        assert e.value.code == -4                      # TSS_E_UNSUPPORTED
        s.close()


@pytest.mark.gpu
def test_limits_leave_no_state_in_the_cached_workspace(fixtures):
    """A limited one-shot solve runs on the workspace an unlimited one cached and caches it again: the next unlimited solve
    (the fused first epoch on that workspace) returns what it returns on an engine that never saw a limit."""
    g = T.WorldGrid(fixtures["ex2"])
    tup = lambda lay: sorted((p.x, p.y, p.definition.width, p.definition.height, int(p.rotated)) for p in lay.platforms().values())
    layouts = []
    for limited in (True, False):
        e = T.Engine(0)
        assert e.solve_upper_bound(g, T.PLATFORMS_DEFAULT, seed=4)[0] == T.SAT     # caches the workspace
        r1, l1 = e.solve_upper_bound(g, T.PLATFORMS_DEFAULT, seed=5)
        if limited:
            r2, l2, obj = e.solve_with_limits(g, T.PLATFORMS_DEFAULT, T.PlatformLimits({P(5, 5): 1, P(3, 3): 1}), seed=6)
            assert r2 == T.SAT and obj == l2.platform_count()
            assert sum(p.definition == P(5, 5) for p in l2.platforms().values()) <= 1 and sum(p.definition == P(3, 3) for p in l2.platforms().values()) <= 1
        r3, l3 = e.solve_upper_bound(g, T.PLATFORMS_DEFAULT, seed=5)
        e.close()
        assert r1 == r3 == T.SAT and tup(l1) == tup(l3)
        layouts.append(tup(l3))
    assert layouts[0] == layouts[1]
