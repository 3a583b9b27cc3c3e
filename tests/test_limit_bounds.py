"""The class-aware fractional lower bound (tss_lower_bound_lp_limits): the LP of csrc/lp.cu with per-type limits kept.

maximise sum_t y_t - sum_j L_j z_j  subject to  sum_{t in reach(p)} y_t - sum_{j: key(p) in class j} z_j <= cost(p) for every
in-bounds placement p,  y, z >= 0

CPU: a HiGHS reference of that LP whose classes agree with the oracle's encoder, against the plain LP and the oracle's optima.
GPU: the entry point without classes against tss_lower_bound_lp, with classes against the reference on every simplex path (the
certificate recomputed in exact fractions), the table's optima, tss_solve_instance with tss_engine_limit_bounds, the REPL's
`-l` loops with --limit-bounds and the error codes."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest
import scipy.optimize
import scipy.sparse

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import golden, rows_to_grid, synth_terrain
from test_lp_reference import _key_dims, _platform_cost, reach_sets
from test_type_limits import _run_repl, oracle_optimum

P = T.PlatformDef
FIXTURES = {k: rows_to_grid(v["grid"]) for k, v in golden("fixtures").items()}
DEFAULT8 = list(O.PLATFORMS_DEFAULT)
GUI_WEIGHTS = {(1, 1): 5, (1, 2): 1, (1, 3): 1, (1, 4): 1, (1, 5): 1, (1, 6): 1, (3, 3): 2, (5, 5): 4}   # crates/gui/src/app.rs:53-62

GRIDS = {"ex1": lambda: FIXTURES["ex1"], "ex2": lambda: FIXTURES["ex2"], "ex3": lambda: FIXTURES["ex3"],
         "random": lambda: synth_terrain(18, 16, seed=7, t=3), "synth32": lambda: synth_terrain(32, 32, seed=1, t=0),
         "rand8x7": lambda: (np.random.default_rng(7).random((7, 8)) < 0.75).astype(np.uint8)}

# (grid, `-l` argument, records, plain LP, class-aware LP): rows where the limits move the optimum above the plain bounds, with
# the LP values HiGHS gives (pinned below on the CPU); the optima come from the oracle's CDCL loop, except on synth32, where that
# loop takes far longer than a test may (there the bound meets ceil(class LP) = 26 and the REPL's loop closes on it)
TABLE = [("ex2", "5:2", {(5, 5): 2}, 4.0, 4.615385), ("ex2", "5:1,1x6:2", {(5, 5): 1, (1, 6): 2}, 4.0, 5.228571),
         ("ex2", "3:1", {(3, 3): 1}, 4.0, 5.0), ("ex2", "1x2:2", {(1, 2): 2}, 4.0, 7.666667),
         ("random", "5:1,3:2", {(5, 5): 1, (3, 3): 2}, 6.0, 7.038462), ("synth32", "3:4", {(3, 3): 4}, 18.965, 25.081),
         ("ex1", "5:0,3:0", {(5, 5): 0, (3, 3): 0}, 1.0, 2.0)]
TABLE_IDS = [f"{g}:{a}" for g, a, *_ in TABLE]
NO_ORACLE = {"synth32"}
# the `-l` loops of test_type_limits.py the plain bounds already close
REPL_CLOSED = [("ex1", "3:1,1x4:2", {(3, 3): 1, (1, 4): 2}), ("ex3", "3:2,1x2:3", {(3, 3): 2, (1, 2): 3})]

_optima = {}


def optimum(name, card):
    key = (name, tuple(sorted(card.items())))
    if key not in _optima:
        _optima[key] = oracle_optimum(GRIDS[name](), DEFAULT8, card)
    return _optima[key]


def class_sets(defs, card):
    """Encoding::with_limits' classes, restated: a limit on type d counts the platforms of every key q that contains a key of
    {d, d^T}; 1x1 and vacuous records (no such key, or a limit of 1024 or more) make none, equal classes merge into the smaller
    limit.  -> (keys, [frozenset of key indices], [limit])"""
    keys = _key_dims(defs)
    sets, lims = [], []
    for (dw, dh), lim in card.items():
        if (dw, dh) == (1, 1) or lim >= 1024:
            continue
        members = frozenset(q for q, kq in enumerate(keys) for k in keys if k in ((dw, dh), (dh, dw)) and k[0] <= kq[0] and k[1] <= kq[1])
        if not members:
            continue
        if members in sets:
            lims[sets.index(members)] = min(lims[sets.index(members)], lim)
        else:
            sets.append(members)
            lims.append(lim)
    return keys, sets, lims


def reduced(defs, card):
    """Defs in a class with limit 0 leave the set, then the classes are taken again -> (defs, keys, sets, limits)"""
    keys, sets, lims = class_sets(defs, card)
    gone = {keys[q] for s, L in zip(sets, lims) if L == 0 for q in s}
    kept = [d for d in defs if tuple(d) not in gone and (d[1], d[0]) not in gone]
    return (kept, *class_sets(kept, card))


class ClassReference:
    """The class-aware LP of one instance, solved by HiGHS."""

    def __init__(self, g, defs, card, weights=None):
        h, w = g.shape
        self.defs, keys, sets, self.limits = reduced(defs, card)
        rs, where = reach_sets(g, self.defs)
        keep = rs.reshape(len(rs), -1).any(1)
        self.where = [p for p, k in zip(where, keep) if k]
        self.A = scipy.sparse.csr_matrix(rs[keep].reshape(int(keep.sum()), h * w).astype(np.int64))
        key_of = [keys.index((kw, kh)) for _, _, kw, kh in self.where]
        self.M = np.array([[1 if k in s else 0 for s in sets] for k in key_of], np.int64).reshape(len(self.where), len(sets))
        self.cost = np.array([1 if weights is None else _platform_cost(kw, kh, weights) for _, _, kw, kh in self.where], np.int64)
        self.tiles = int(g.sum())
        max_cost = max(1, max(_platform_cost(kw, kh, weights) for kw, kh in keys) if weights else 1)
        scale = float(1 << 20)
        while scale * max_cost > float(1 << 30):
            scale *= 0.5
        self.scale = scale
        cols = np.flatnonzero(g.reshape(-1))
        J = len(self.limits)
        A = scipy.sparse.hstack([self.A[:, cols], scipy.sparse.csr_matrix(-self.M)]).tocsr()
        c = np.concatenate([-np.ones(len(cols)), np.array(self.limits, float)])
        res = scipy.optimize.linprog(c, A_ub=A, b_ub=self.cost.astype(float), bounds=(0, None), method="highs")
        assert res.status == 0, res.message
        self.lp = -res.fun
        # floor(y * scale) loses < 1 / scale per tile; floor(z * scale) raises a net load by < 1 per class of the key, so
        # the ratio V / load by at most J * lp / scale
        self.tol = (self.tiles + J * (self.lp + 1)) / scale + 1e-6 * self.lp

    def certified(self, weights, class_weights):
        """-> (v, max net load): v = min over placements with a positive net load of V * cost / load in exact fractions, 0 if
        V <= 0 or nothing carries load"""
        k = np.asarray(weights, np.int64).reshape(-1)
        zeta = np.asarray(class_weights, np.int64)[: len(self.limits)]
        loads = self.A @ k - self.M @ zeta
        V = int(k.sum()) - int(np.dot(self.limits, zeta)) if len(self.limits) else int(k.sum())
        carrying = np.flatnonzero(loads > 0)
        if len(carrying) == 0:
            return Fraction(0), 0, V
        v = min(Fraction(V * int(self.cost[i]), int(loads[i])) for i in carrying) if V > 0 else Fraction(0)
        return v, int(loads.max()), V


def plain_lp(g, defs):
    h, w = g.shape
    rs, _ = reach_sets(g, defs)
    A = rs.reshape(len(rs), -1)
    A = A[A.any(1)][:, np.flatnonzero(g.reshape(-1))].astype(float)
    res = scipy.optimize.linprog(-np.ones(A.shape[1]), A_ub=scipy.sparse.csr_matrix(A), b_ub=np.ones(len(A)), bounds=(0, None), method="highs")
    return -res.fun


_refs = {}


def reference(name, card, defs=None, weights=None):
    key = (name, tuple(sorted(card.items())), tuple(defs or ()), tuple(sorted((weights or {}).items())))
    if key not in _refs:
        _refs[key] = ClassReference(GRIDS[name](), list(defs or DEFAULT8), card, weights)
    return _refs[key]


# ---------------------------------------------------------------------------------------------------------- CPU tests
@pytest.mark.parametrize("card", [c for _, _, c, *_ in TABLE] + [c for *_, c in REPL_CLOSED] + [{(1, 6): 4, (6, 1): 2, (2, 2): 1, (4, 4): 1024}])
def test_reference_classes_match_the_oracle_encoder_and_the_engine(card):
    """A platform of key q alone is a propagation conflict of the oracle's CNF under with_limits({d: 0}) exactly when q is in the
    reference's class of d; the reference's classes (and their merging) are tss_card_limit_classes'."""
    grid = np.ones((8, 8), np.uint8)
    enc = O.Encoding(DEFAULT8, grid)
    for d in card:
        cnf = enc.with_limits(card_limits={d: 0})
        _, sets, _ = class_sets(DEFAULT8, {d: 0})
        members = sets[0] if sets else frozenset()
        for qi in range(len(enc.dims)):
            a = np.full(cnf.n_vars + 1, 2, np.uint8)
            a[enc.plat_var[0, qi]] = 1
            _, conflict, _ = cnf.propagate(a)
            assert (conflict >= 0) == (qi in members), (d, enc.dims[qi])
    keys, sets, lims = class_sets(DEFAULT8, card)
    ekeys, emask, elim = T.card_limit_classes([P(*d) for d in DEFAULT8], {P(*d): v for d, v in card.items()})
    assert ekeys == keys and elim == lims
    assert [frozenset(q for q in range(len(keys)) if (emask[q] >> j) & 1) for j in range(len(lims))] == sets


@pytest.mark.parametrize("name,arg,card,plain,pinned", TABLE, ids=TABLE_IDS)
def test_class_lp_dominates_the_plain_lp_and_stays_below_the_optimum(name, arg, card, plain, pinned):
    ref = reference(name, card)
    assert abs(ref.lp - pinned) < 1e-3 and abs(plain_lp(GRIDS[name](), DEFAULT8) - plain) < 1e-3, (ref.lp, pinned)
    assert ref.lp >= plain - 1e-9
    if name not in NO_ORACLE:
        assert math.ceil(ref.lp - ref.tol) <= optimum(name, card)


# ---------------------------------------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def _select_path(monkeypatch, path):
    if path == "single":
        monkeypatch.setenv("TSS_LP_SINGLE_CTA", "1")
    else:
        monkeypatch.delenv("TSS_LP_SINGLE_CTA", raising=False)


def _lp(eng, name, card=None, defs=None, weights=None, **kw):
    defs = [P(*d) for d in (defs or DEFAULT8)]
    wts = None if weights is None else {P(*d): v for d, v in weights.items()}
    lim = None if card is None else {P(*d): v for d, v in card.items()}
    return eng.lower_bound_lp(T.WorldGrid(GRIDS[name]() if name in GRIDS else NO_CLASS_GRIDS[name]()), defs, weights=wts, limits=lim, **kw)


NO_CLASS_GRIDS = {"rect21": lambda: np.ones((21, 21), np.uint8), "rect16": lambda: np.ones((16, 16), np.uint8)}
# (grid, defs, weights, path) of test_lp_reference.CASES: the cluster, the grid kernel and the one-CTA kernel
NO_CLASS_CASES = [("ex1", None, None, "cluster"), ("ex2", [(1, 1)], None, "cluster"), ("ex1", None, GUI_WEIGHTS, "cluster"),
                  ("rect21", [(1, 1)], None, "grid"), ("ex2", None, None, "grid"),
                  ("ex2", [(1, 1)], None, "single"), ("rect16", [(1, 1)], None, "single")]


@pytest.mark.gpu
@pytest.mark.parametrize("name,defs,weights,path", NO_CLASS_CASES, ids=[f"{c[0]}/{c[3]}/{'gui' if c[2] else len(c[1] or DEFAULT8)}" for c in NO_CLASS_CASES])
def test_no_class_is_the_plain_lp(eng, monkeypatch, name, defs, weights, path):
    """No records, a 1x1 record, vacuous records: tss_lower_bound_lp_limits returns what tss_lower_bound_lp returns, bit for bit,
    run to optimality and stopped at a target."""
    _select_path(monkeypatch, path)
    for kw in (dict(), dict(target=3)):
        want = _lp(eng, name, None, defs, weights, **kw)
        for card in ({}, {(1, 1): 5}, {(2, 2): 1, (5, 5): 2000, (4, 6): 0}):
            got = _lp(eng, name, card, defs, weights, **kw)
            assert not got["class_weights"].any()
            for k in ("bound", "total", "max_load", "pivots", "optimal", "constraints"):
                assert got[k] == want[k], (k, card, got[k], want[k])
            assert np.array_equal(got["weights"], want["weights"])


# (grid, records, defs, weights, path) with classes
CLASS_CASES = [("ex1", {(3, 3): 1, (1, 4): 2}, None, None, "cluster"), ("ex3", {(3, 3): 2, (1, 2): 3}, None, None, "cluster"),
               ("rand8x7", {(3, 3): 1}, [(1, 1), (1, 3), (3, 3)], None, "cluster"), ("ex1", {(5, 5): 1}, None, GUI_WEIGHTS, "cluster"),
               ("ex2", {(5, 5): 2}, None, None, "grid"), ("ex2", {(5, 5): 1, (1, 6): 2}, None, None, "grid"), ("ex2", {(1, 2): 2}, None, None, "grid"),
               ("ex2", {(5, 5): 2}, None, None, "single"), ("ex1", {(5, 5): 0, (3, 3): 0}, None, None, "single"), ("ex3", {(3, 3): 2, (1, 2): 3}, None, None, "single")]
CLASS_IDS = [f"{g}/{','.join(f'{a}x{b}:{v}' for (a, b), v in c.items())}/{'gui' if w else len(d or DEFAULT8)}/{p}" for g, c, d, w, p in CLASS_CASES]


def _check_certificate(ref, r):
    """The bound is ceil(v) for the weights the call reports, v recomputed from the reference's placements in exact fractions"""
    k, z = r["weights"].astype(np.int64), r["class_weights"]
    assert (k >= 0).all() and (z >= 0).all() and not z[len(ref.limits):].any()
    v, max_load, V = ref.certified(k, z)
    assert r["total"] == V
    assert r["bound"] == math.ceil(v), (r["bound"], v)
    if (ref.cost == 1).all():
        assert r["max_load"] == max_load
    assert v <= ref.lp * (1 + 1e-6) + 1e-12, (v, ref.lp)    # weak duality
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("name,card,defs,weights,path", CLASS_CASES, ids=CLASS_IDS)
def test_class_lp_reaches_the_reference_optimum(eng, monkeypatch, name, card, defs, weights, path):
    """Run to optimality the simplex reaches the class LP's optimum up to the resolution of the integer weights, and the reported
    bound is the exact certificate of the weights it reports; with a target it stops early and still reaches min(target, optimum)."""
    _select_path(monkeypatch, path)
    ref = reference(name, card, defs, weights)
    r = _lp(eng, name, card, defs, weights)
    v = _check_certificate(ref, r)
    assert r["optimal"], r["pivots"]
    assert v >= ref.lp - ref.tol, (float(v), ref.lp, ref.tol)
    low, top = math.ceil(ref.lp - ref.tol), math.ceil(ref.lp + 1e-6)
    assert low <= r["bound"] <= top
    again = _lp(eng, name, card, defs, weights)
    assert np.array_equal(again["weights"], r["weights"]) and np.array_equal(again["class_weights"], r["class_weights"])
    for t in range(1, top + 2):
        rt = _lp(eng, name, card, defs, weights, target=t)
        _check_certificate(ref, rt)
        assert min(t, low) <= rt["bound"] <= top, (t, rt["bound"], ref.lp, rt["pivots"])
    r5 = _lp(eng, name, card, defs, weights, max_pivots=5)
    assert r5["pivots"] <= 5
    _check_certificate(ref, r5)


@pytest.mark.gpu
@pytest.mark.parametrize("name,arg,card,plain,pinned", TABLE, ids=TABLE_IDS)
def test_class_bound_is_the_optimum(eng, monkeypatch, name, arg, card, plain, pinned):
    monkeypatch.delenv("TSS_LP_SINGLE_CTA", raising=False)
    ref = reference(name, card)
    want = math.ceil(ref.lp - ref.tol) if name in NO_ORACLE else optimum(name, card)
    r = _lp(eng, name, card)
    _check_certificate(ref, r)
    assert r["bound"] == want, (r["bound"], want, r["pivots"])
    assert _lp(eng, name)["bound"] < want                     # the plain LP does not close it
    assert _lp(eng, name, card, target=want)["bound"] == want


def _instance(eng, grid, card):
    from timberborn_support_solver_b200 import _lib
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, T.WorldGrid(grid))
    cnf = enc.with_limits(T.PlatformLimits({P(*d): v for d, v in card.items()}))
    dev = eng.upload_cnf(cnf)
    lits, offs = np.ascontiguousarray(cnf.lits, np.int32), np.ascontiguousarray(cnf.offsets, np.uint32)
    info, h = _lib.InstanceInfo(), C.c_void_p()
    assert eng.lib.tss_instance_find(lits.ctypes.data_as(C.POINTER(C.c_int32)), offs.ctypes.data_as(C.POINTER(C.c_uint32)), cnf.n_clauses, cnf.n_vars,
                                     C.byref(h), C.byref(info), None, 0) == _lib.TSS_SAT
    return enc, cnf, dev, h, info


def _solve_instance(eng, inst, give_up):
    _, cnf, dev, h, info = inst
    a = np.full(cnf.n_vars + 1, 2, np.uint8)
    eng.clear_interrupt()
    return eng.lib.tss_solve_instance(eng._h, dev._h, h, C.byref(info), None, 1, give_up, a.ctypes.data_as(C.POINTER(C.c_uint8))), a


@pytest.mark.gpu
@pytest.mark.parametrize("row", [0, 2, 6], ids=[TABLE_IDS[i] for i in (0, 2, 6)])
def test_solve_instance_certifies_limited_instances(row):
    """With tss_engine_limit_bounds: UNSAT one below the optimum, SAT at it with a witness of the oracle's CNF.  Switched off, or
    with the bound-based answers off: UNKNOWN below the optimum, as before."""
    from timberborn_support_solver_b200 import _lib
    name, _, card, _, _ = TABLE[row]
    grid, want = GRIDS[name](), optimum(name, card)
    e = T.Engine(0)
    try:
        below = _instance(e, grid, {**card, (1, 1): want - 1})
        assert _solve_instance(e, below, 4096)[0] == _lib.TSS_UNKNOWN          # off by default
        e.limit_bounds(True)
        assert _solve_instance(e, below, 4096)[0] == _lib.TSS_UNSAT
        assert _solve_instance(e, below, 4096)[0] == _lib.TSS_UNSAT            # (the cached bound)
        at = _instance(e, grid, {**card, (1, 1): want})
        rc, a = _solve_instance(e, at, 0)
        assert rc == _lib.TSS_SAT
        assert O.Encoding(O.PLATFORMS_DEFAULT, grid).with_limits(card_limits={**card, (1, 1): want}).count_falsified(a)[0] == 0
        assert e.lib.tss_engine_certified_unsat(e._h, 0) == 0
        assert _solve_instance(e, below, 4096)[0] == _lib.TSS_UNKNOWN
        assert e.lib.tss_engine_certified_unsat(e._h, 1) == 0
        e.limit_bounds(False)
        assert _solve_instance(e, below, 4096)[0] == _lib.TSS_UNKNOWN
        for inst in (below, at):
            e.lib.tss_encoding_destroy(inst[3])
    finally:
        e.close()


# the table's loops and the closed ones (not synth32: a loop there that missed the optimum would leave 32x32 to the exact solver)
REPL_ROWS = [(g, a, c) for g, a, c, *_ in TABLE if g not in NO_ORACLE] + REPL_CLOSED


@pytest.mark.gpu
@pytest.mark.parametrize("name,arg,card", REPL_ROWS, ids=[f"{n}:{a}" for n, a, _ in REPL_ROWS])
def test_repl_limit_loop_ends_on_the_class_bound(tmp_path, name, arg, card):
    """The loop reaches the oracle's optimum and its last UNSAT comes from the class-aware bound (lower_bound = the optimum).  The
    exact solver is asked at most once, for a layout the search missed, never for the proof."""
    want = optimum(name, card)
    text, f, counts = _run_repl(tmp_path, GRIDS[name](), "-l", arg, "--seed", "3", "--limit-bounds")
    assert int(f["best"]) == want and counts[-1] == want, (text, want)
    assert 'verdict="optimal (lower bound)"' in text and int(f["lower_bound"]) == want, text
    assert int(f["exact_solves"]) <= 1 and "FAILED" not in text, text
    assert text.count("Solution validation OK (exact)") == int(f["exact_solves"]), text


@pytest.mark.gpu
def test_repl_no_lower_bound_wins_over_limit_bounds(tmp_path):
    name, arg, card = "ex2", "5:2", {(5, 5): 2}
    text, f, _ = _run_repl(tmp_path, GRIDS[name](), "-l", arg, "--seed", "3", "--limit-bounds", "--no-lower-bound")
    assert int(f["best"]) == optimum(name, card) and int(f["exact_solves"]) == 1 and int(f["lower_bound"]) == -1, text


@pytest.mark.gpu
def test_solver_loop_with_limit_bounds(eng):
    name, card = "ex2", {(5, 5): 2}
    grid = T.WorldGrid(GRIDS[name]())
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, grid)
    out = T.solver_loop(T.Project(T.World(grid)), enc, T.PlatformLimits({P(*d): v for d, v in card.items()}), eng, seed=3, limit_bounds=True)
    assert out["proved_optimal"] and out["best"].platform_count() == optimum(name, card) == out["lower_bound"]
    assert out["steps"][-1]["source"] == "lower bound"


@pytest.mark.gpu
def test_limit_bound_error_codes(eng):
    big = T.WorldGrid(synth_terrain(48, 48, seed=2, t=1))
    defs = list(T.PLATFORMS_DEFAULT)
    with pytest.raises(T.TssError) as e:
        eng.lower_bound_lp(big, defs, limits={P(5, 5): 3}, max_pivots=50)
    assert e.value.code == -4                                   # TSS_E_UNSUPPORTED
    vac = eng.lower_bound_lp(big, defs, limits={P(2, 2): 1, P(1, 1): 9}, max_pivots=50)
    plain = eng.lower_bound_lp(big, defs, max_pivots=50)
    assert vac["bound"] == plain["bound"] and np.array_equal(vac["weights"], plain["weights"]) and not vac["class_weights"].any()
    for g in (big, T.WorldGrid(FIXTURES["ex1"])):
        with pytest.raises(T.TssError) as e:
            eng.lower_bound_lp(g, defs, limits={P(3, 3): -1})
        assert e.value.code == -1                               # TSS_E_INVALID
