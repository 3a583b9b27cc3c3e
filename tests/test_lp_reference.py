"""The fractional lower bound (csrc/lp.cu) against a reference solve of the same LP.

maximise sum_t y_t  subject to  sum_{t in reach(p)} y_t <= cost(p) for every in-bounds placement p,  y >= 0

The reference builds every placement's reach set in numpy (checked against the oracle's validate) and solves the LP with
HiGHS.  On the device the certificate is exact whatever the simplex does, so the tests below check what the certificate
cannot: that the simplex reaches the LP optimum, on each of the three simplex kernels, up to the resolution of the integer
weights it reports."""
import math
from fractions import Fraction

import numpy as np
import pytest
import scipy.optimize
import scipy.sparse

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import golden, rows_to_grid, synth_terrain

GUI_WEIGHTS = {(1, 1): 5, (1, 2): 1, (1, 3): 1, (1, 4): 1, (1, 5): 1, (1, 6): 1, (3, 3): 2, (5, 5): 4}   # crates/gui/src/app.rs:53-62
B200_SMS = 148                            # the grid kernel runs one CTA per SM, at most (m + 3) / 4 of them
MAX_COLS = 1024                           # lp.cu: ceiling tiles of a 32x32 grid


def _key_dims(defs):
    out = []
    for d in defs:      # dims keys: defs order, unflipped then flipped (src/encoder.rs:121-130)
        for dims in ((d[0], d[1]), (d[1], d[0])):
            if dims not in out:
                out.append(dims)
    return out


def _platform_cost(kw, kh, weights):
    """what PlatformLayout::total_weight charges one platform: the weights of every def that fits inside its def (platform_layout.rs:174-183)"""
    cw, ch = min(kw, kh), max(kw, kh)
    return sum(v for (dw, dh), v in weights.items() if min(dw, dh) <= cw and max(dw, dh) <= ch)


def _dilate(X, C):
    Y = X.copy()
    Y[:, 1:] |= X[:, :-1]
    Y[:, :-1] |= X[:, 1:]
    Y[:, :, 1:] |= X[:, :, :-1]
    Y[:, :, :-1] |= X[:, :, 1:]
    return Y & C


def reach_sets(g, defs):
    """Every in-bounds placement of every dims key (defs order, key by key, anchors row-major) -> (bool[P, h, w] reach sets,
    [(x, y, kw, kh)] placements).  reach = footprint & ceiling, then three 4-neighbour dilations each masked by the ceiling."""
    h, w = g.shape
    C = g.astype(bool)[None]
    sets, where = [], []
    for kw, kh in _key_dims(defs):
        anchors = [(x, y) for y in range(h - kh + 1) for x in range(w - kw + 1)]
        if not anchors:
            continue
        X = np.zeros((len(anchors), h, w), bool)
        for i, (x, y) in enumerate(anchors):
            X[i, y:y + kh, x:x + kw] = True
        X &= C
        for _ in range(3):
            X = _dilate(X, C)
        sets.append(X)
        where += [(x, y, kw, kh) for x, y in anchors]
    return np.concatenate(sets), where


class Reference:
    """The LP of one instance, solved by HiGHS: the constraint rows are the placements whose footprint covers ceiling."""

    def __init__(self, g, defs, weights=None):
        h, w = g.shape
        sets, where = reach_sets(g, defs)
        keep = sets.reshape(len(sets), -1).any(1)
        self.where = [p for p, k in zip(where, keep) if k]
        self.A = scipy.sparse.csr_matrix(sets[keep].reshape(int(keep.sum()), h * w).astype(np.int64))
        self.cost = np.array([1 if weights is None else _platform_cost(kw, kh, weights) for _, _, kw, kh in self.where], np.int64)
        self.rows = len(self.where)
        self.tiles = int(g.sum())
        self.max_cost = max(1, max(_platform_cost(kw, kh, weights) for kw, kh in _key_dims(defs)) if weights else 1)
        scale = float(1 << 20)                 # lp.cu: integer weights floor(y * scale) stay below 2^30
        while scale * self.max_cost > float(1 << 30):
            scale *= 0.5
        self.scale = scale
        cols = np.flatnonzero(g.reshape(-1))
        res = scipy.optimize.linprog(-np.ones(len(cols)), A_ub=self.A[:, cols], b_ub=self.cost.astype(float), bounds=(0, None), method="highs")
        assert res.status == 0, res.message
        self.lp = -res.fun
        self.tol = self.tiles / self.scale + 1e-6 * self.lp   # floor(y * scale) loses < 1 / scale per tile

    def certified(self, weights):
        """-> (v, max load): v = min over placements with load > 0 of total * cost / load, exact (0 if nothing carries load)"""
        wts = np.asarray(weights, np.int64).reshape(-1)
        loads = self.A @ wts
        total = int(wts.sum())
        carrying = np.flatnonzero(loads > 0)
        if len(carrying) == 0:
            return Fraction(0), 0
        return min(Fraction(total * int(self.cost[i]), int(loads[i])) for i in carrying), int(loads.max())


# --------------------------------------------------------------------------------------------------------- the instances
FIXTURES = {k: rows_to_grid(v["grid"]) for k, v in golden("fixtures").items()}
README = rows_to_grid(golden("readme_layouts")["terrain"])
DEFS_1X1 = [(1, 1)]
DEFS_DEFAULT = list(O.PLATFORMS_DEFAULT)
DEFS_133 = [(1, 1), (1, 3), (3, 3)]


def _corridor():
    return np.ones((1, 32), np.uint8)


def _islands():
    g = np.zeros((1, 32), np.uint8)
    g[0, 0] = g[0, 31] = 1
    return g


def _sparse():
    return (np.random.default_rng(21).random((32, 32)) < 0.12).astype(np.uint8)


def _rand8x7():
    return (np.random.default_rng(7).random((7, 8)) < 0.75).astype(np.uint8)


def _rand9x10():
    return (np.random.default_rng(13).random((10, 9)) < 0.8).astype(np.uint8)


GRIDS = {
    "1x1": lambda: np.ones((1, 1), np.uint8), "strip1x3": lambda: np.ones((1, 3), np.uint8), "islands": _islands, "corridor": _corridor,
    "ex1": lambda: FIXTURES["ex1"], "ex2": lambda: FIXTURES["ex2"], "ex3": lambda: FIXTURES["ex3"], "readme": lambda: README,
    "rect16": lambda: np.ones((16, 16), np.uint8), "rect19": lambda: np.ones((19, 19), np.uint8), "rect21": lambda: np.ones((21, 21), np.uint8),
    "rect24": lambda: np.ones((24, 24), np.uint8), "rect32": lambda: np.ones((32, 32), np.uint8),
    "rand20x14": lambda: synth_terrain(20, 14, seed=3, t=1), "synth27x25": lambda: synth_terrain(27, 25, seed=2, t=0),
    "synth32": lambda: synth_terrain(32, 32, seed=1, t=0), "synth32x31": lambda: synth_terrain(32, 31, seed=4, t=0),
    "synth31x32": lambda: synth_terrain(31, 32, seed=5, t=0), "sparse32": _sparse, "rand8x7": _rand8x7, "rand9x10": _rand9x10,
}
PSETS = {"1x1": (DEFS_1X1, None), "default8": (DEFS_DEFAULT, None), "133": (DEFS_133, None), "gui": (DEFS_DEFAULT, GUI_WEIGHTS),
         "w4096": (DEFS_133, {(1, 1): 1000, (1, 3): 96, (3, 3): 3000}),        # 3x3 key costs 4096: scale 2^18
         "w3907": ([(1, 1), (1, 2), (2, 2)], {(1, 1): 7, (1, 2): 900, (2, 2): 3000})}

# (grid, platform set, kernel path): the path is what lp_path() predicts for the default launch, or "single" where the test forces the
# one-CTA kernel (TSS_LP_SINGLE_CTA=1)
CASES = [
    ("1x1", "1x1", "cluster"), ("strip1x3", "1x1", "cluster"), ("islands", "1x1", "cluster"), ("corridor", "1x1", "cluster"),
    ("ex1", "1x1", "cluster"), ("ex3", "1x1", "cluster"), ("ex2", "1x1", "cluster"), ("readme", "1x1", "cluster"),
    ("rect16", "1x1", "cluster"), ("rand20x14", "1x1", "cluster"), ("rect19", "1x1", "cluster"), ("sparse32", "1x1", "cluster"),
    ("ex1", "default8", "cluster"), ("ex3", "default8", "cluster"), ("rand8x7", "133", "cluster"),
    ("ex1", "gui", "cluster"), ("ex3", "gui", "cluster"), ("rand9x10", "w4096", "cluster"), ("rand8x7", "w3907", "cluster"),
    ("rect21", "1x1", "grid"), ("synth27x25", "1x1", "grid"), ("synth32", "1x1", "grid"), ("rect32", "1x1", "grid"),
    ("synth32x31", "1x1", "grid"), ("synth31x32", "133", "grid"), ("sparse32", "default8", "grid"),
    ("ex2", "default8", "grid"), ("rect24", "default8", "grid"), ("rect32", "default8", "grid"),
    ("ex1", "1x1", "single"), ("ex3", "1x1", "single"), ("ex2", "1x1", "single"), ("readme", "1x1", "single"), ("rect16", "1x1", "single"),
    ("rand20x14", "1x1", "single"), ("corridor", "1x1", "single"), ("ex2", "default8", "single"), ("rect32", "1x1", "single"),
]
CASE_IDS = [f"{g}/{p}/{path}" for g, p, path in CASES]

_refs = {}


def reference(grid_name, pset):
    if (grid_name, pset) not in _refs:
        defs, weights = PSETS[pset]
        _refs[(grid_name, pset)] = Reference(GRIDS[grid_name](), defs, weights)
    return _refs[(grid_name, pset)]


_rows = {}


def reference_rows(grid_name, pset):
    """(constraints, ceiling tiles) without solving the LP"""
    if (grid_name, pset) not in _rows:
        g = GRIDS[grid_name]()
        sets, _ = reach_sets(g, PSETS[pset][0])
        _rows[(grid_name, pset)] = (int(sets.reshape(len(sets), -1).any(1).sum()), int(g.sum()))
    return _rows[(grid_name, pset)]


def lp_path(m, n, sms=B200_SMS):
    """The kernel lp_run launches for a tableau of m constraints x n tiles (lp.cu: the cluster when its shared memory fits 200 KB,
    else the cooperative grid kernel on G CTAs) -> ("cluster", rows per CTA) or ("grid", G)."""
    rows_per, ld = (m + 7) // 8, n + 1
    cl_smem = 8 * (rows_per * ld + 2 * ld + rows_per + 2 * 8 * ld) + 16 * 2 * 8 + 4 * (m + n)
    if cl_smem <= 200 * 1024:
        return "cluster", rows_per
    return "grid", max(1, min(sms, (m + 3) // 4))


# ---------------------------------------------------------------------------------------------------------- CPU tests
def test_reference_reach_sets_match_validate_and_lp_values_are_pinned():
    """The numpy reach sets are validate()'s rule (platform_layout.rs:85-149) for one platform alone, placement by placement, and
    the reference LP reproduces the LP values of the named instances."""
    for g, defs in ((FIXTURES["ex1"], DEFS_DEFAULT), (FIXTURES["ex3"], DEFS_DEFAULT), (_rand8x7(), DEFS_133), (_corridor(), DEFS_1X1)):
        sets, where = reach_sets(g, defs)
        assert len(where) == sum((g.shape[1] - kw + 1) * (g.shape[0] - kh + 1) for kw, kh in _key_dims(defs))
        for X, (x, y, kw, kh) in zip(sets, where):
            v = O.validate(g, [(x, y, min(kw, kh), max(kw, kh), int(kw > kh))])
            assert not v.out_of_bounds
            assert np.array_equal(X, (g & (1 - v.unsupported)).astype(bool)), (x, y, kw, kh)
    pinned = {("ex2", "1x1"): 13.2, ("readme", "1x1"): 13.131754706, ("rect16", "1x1"): 13.468448404, ("ex2", "default8"): 4.0, ("corridor", "1x1"): 5.0}
    for key, want in pinned.items():
        assert abs(reference(*key).lp - want) < 1e-6, (key, reference(*key).lp)
    assert reference("ex2", "default8").rows == 2968 and reference("ex2", "1x1").rows == 236 and reference("readme", "1x1").rows == 240


def test_case_list_covers_every_simplex_path():
    """Each kernel runs on at least three cases, and on the edges where its indexing changes: a cluster with CTAs that own no rows,
    a row count not a multiple of 8 and more than 32 rows per CTA; a grid below the SM count with a ragged last CTA and grids on
    every SM; the one-CTA kernel up to MAX_COLS columns."""
    paths = {"cluster": [], "grid": [], "single": []}
    for g, p, path in CASES:
        ref = reference_rows(g, p)
        predicted = lp_path(*ref)
        if path != "single":
            assert predicted[0] == path, (g, p, ref, predicted)
        paths[path].append((g, p, ref, predicted))
    assert all(len(v) >= 3 for v in paths.values())
    cl = paths["cluster"]
    assert any(m < 8 for _, _, (m, _), _ in cl)
    assert any(m % 8 for _, _, (m, _), _ in cl)
    assert any(rows_per > 32 for _, _, _, (_, rows_per) in cl)
    gr = paths["grid"]
    assert any(G < B200_SMS and m % G for _, _, (m, _), (_, G) in gr)
    assert sum(G == B200_SMS for _, _, _, (_, G) in gr) >= 3
    assert any(n == MAX_COLS for _, _, (_, n), _ in paths["single"]) and any(n == MAX_COLS for _, _, (_, n), _ in gr)



# ---------------------------------------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def _api_args(pset):
    defs, weights = PSETS[pset]
    return [T.PlatformDef(*d) for d in defs], None if weights is None else {T.PlatformDef(*d): v for d, v in weights.items()}


def _select_path(monkeypatch, path):
    if path == "single":
        monkeypatch.setenv("TSS_LP_SINGLE_CTA", "1")
    else:
        monkeypatch.delenv("TSS_LP_SINGLE_CTA", raising=False)


def _check_certificate(ref, r):
    """The reported bound is ceil(v) for the weights it reports, v recomputed from the reference's placements in exact
    arithmetic (a placement missing on the device would show here) -> v"""
    wts = r["weights"].astype(np.int64)
    assert (wts >= 0).all() and int(wts.sum()) == r["total"]
    v, max_load = ref.certified(wts)
    assert r["bound"] == math.ceil(v), (r["bound"], v)
    if ref.max_cost == 1 and (ref.cost == 1).all():
        assert r["max_load"] == max_load
    assert r["constraints"] == ref.rows                  # the device's compaction keeps exactly the placements that cover ceiling
    assert v <= ref.lp * (1 + 1e-6) + 1e-12, (v, ref.lp)   # weak duality: above the optimum means the reference or the certificate is wrong
    return v


def _lower_bound_lp(eng, grid_name, pset, **kw):
    defs, weights = _api_args(pset)
    return eng.lower_bound_lp(T.WorldGrid(GRIDS[grid_name]()), defs, weights=weights, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("grid_name,pset,path", CASES, ids=CASE_IDS)
def test_lp_reaches_the_reference_optimum(eng, monkeypatch, grid_name, pset, path):
    """Run to optimality, the simplex reaches the LP optimum up to the resolution of the integer weights (n / scale): a simplex
    that stops early is caught here even where ceil() lands on the same integer."""
    _select_path(monkeypatch, path)
    ref = reference(grid_name, pset)
    r = _lower_bound_lp(eng, grid_name, pset)
    v = _check_certificate(ref, r)
    assert r["optimal"], r["pivots"]
    assert v >= ref.lp - ref.tol, (float(v), ref.lp, ref.tol, r["pivots"])
    assert math.ceil(ref.lp - ref.tol) <= r["bound"] <= math.ceil(ref.lp + 1e-6)
    if grid_name == "corridor":
        assert r["bound"] == 5                            # an interval LP: its optimum is integral
    again = _lower_bound_lp(eng, grid_name, pset)
    assert np.array_equal(again["weights"], r["weights"]) and again["pivots"] == r["pivots"]


def _targets(lp):
    top = math.ceil(lp) + 1
    if top <= 80:
        return list(range(1, top + 1))
    return sorted(set(range(1, 11)) | set(int(t) for t in np.linspace(1, top, 30)) | set(range(top - 20, top + 1)))


@pytest.mark.gpu
@pytest.mark.parametrize("grid_name,pset,path", CASES, ids=CASE_IDS)
def test_lp_early_stops_keep_the_bound(eng, monkeypatch, grid_name, pset, path):
    """With a target the simplex may stop once the objective has passed target - 1 with a margin for rounding, and reruns to
    optimality when the certificate falls short: the bound reaches the target or the optimum, whichever is lower.  An iteration
    cap only weakens the bound; the certificate stays exact."""
    _select_path(monkeypatch, path)
    ref = reference(grid_name, pset)
    low, top = math.ceil(ref.lp - ref.tol), math.ceil(ref.lp + 1e-6)
    for t in _targets(ref.lp):
        r = _lower_bound_lp(eng, grid_name, pset, target=t)
        _check_certificate(ref, r)
        assert min(t, low) <= r["bound"] <= top, (t, r["bound"], ref.lp, r["pivots"], r["optimal"])
    for k in (1, 5, 50):
        r = _lower_bound_lp(eng, grid_name, pset, max_pivots=k)
        assert r["pivots"] <= k
        _check_certificate(ref, r)


@pytest.mark.gpu
def test_lp_scratch_reuse_matches_fresh_engines(monkeypatch):
    """lp_run reuses grow-only scratch slots across calls: the case list forwards then backwards on one engine gives the weights
    of a fresh engine per case."""
    monkeypatch.delenv("TSS_LP_SINGLE_CTA", raising=False)
    cases = [(g, p) for g, p, path in CASES if path != "single"]
    fresh = {}
    for g, p in cases:
        e = T.Engine(0)
        fresh[(g, p)] = _lower_bound_lp(e, g, p)["weights"]
        e.close()
    e = T.Engine(0)
    for g, p in cases + cases[::-1]:
        assert np.array_equal(_lower_bound_lp(e, g, p)["weights"], fresh[(g, p)]), (g, p)
    e.close()


@pytest.mark.gpu
def test_lp_weight_objective_edges(eng, monkeypatch):
    """A platform that costs nothing: every tile lies in the reach of its own 1x1 placement, so the LP optimum and the bound are 0.
    Key costs above 4096 (here a 3x3 key: 1 + 4096) are rejected."""
    monkeypatch.delenv("TSS_LP_SINGLE_CTA", raising=False)
    g = _rand9x10()
    free = {(1, 1): 0, (1, 3): 2, (3, 3): 5}
    assert abs(Reference(g, DEFS_133, free).lp) < 1e-9
    defs = [T.PlatformDef(*d) for d in DEFS_133]
    r = eng.lower_bound_lp(T.WorldGrid(g), defs, weights={T.PlatformDef(*d): v for d, v in free.items()})
    assert r["bound"] == 0 and r["total"] == 0 and not r["weights"].any()
    with pytest.raises(T.TssError):
        eng.lower_bound_lp(T.WorldGrid(g), defs, weights={T.PlatformDef(1, 1): 1, T.PlatformDef(3, 3): 4096})
