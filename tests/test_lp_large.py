"""The fractional lower bound on grids larger than 32x32 (csrc/lp_big.cu: a first-order method instead of the simplex, the same
integer certificate).

The reference here builds every placement's reach from its (kw + 6) x (kh + 6) window of the ceiling (three masked dilations of the
footprint cannot leave it), checked against test_lp_reference.reach_sets on small grids, recomputes each certificate exactly and
solves the LP with HiGHS for the quality bars."""
import math
from fractions import Fraction

import numpy as np
import pytest
import scipy.optimize
import scipy.sparse

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import synth_terrain
from test_lp_reference import GUI_WEIGHTS, _key_dims, _platform_cost, reach_sets

DEFS_1X1 = [(1, 1)]
DEFS_DEFAULT = list(O.PLATFORMS_DEFAULT)
HALO = 3


def window_reach(g, defs):
    """-> list of (key dims, anchors [(x, y)], bool[P, kh + 6, kw + 6] reach windows) for every in-bounds placement of every key.
    Window row r = grid row y - 3 + r, column c = grid column x - 3 + c."""
    h, w = g.shape
    pad = np.zeros((h + 2 * HALO + 6, w + 2 * HALO + 6), bool)
    pad[HALO:HALO + h, HALO:HALO + w] = g.astype(bool)
    out = []
    for kw, kh in _key_dims(defs):
        ys, xs = np.mgrid[0:h - kh + 1, 0:w - kw + 1]
        ys, xs = ys.reshape(-1), xs.reshape(-1)
        if len(xs) == 0:
            continue
        rr, cc = np.mgrid[0:kh + 2 * HALO, 0:kw + 2 * HALO]
        Cw = pad[ys[:, None, None] + rr[None], xs[:, None, None] + cc[None]]
        X = np.zeros_like(Cw)
        X[:, HALO:HALO + kh, HALO:HALO + kw] = Cw[:, HALO:HALO + kh, HALO:HALO + kw]
        for _ in range(HALO):
            Y = X.copy()
            Y[:, 1:] |= X[:, :-1]
            Y[:, :-1] |= X[:, 1:]
            Y[:, :, 1:] |= X[:, :, :-1]
            Y[:, :, :-1] |= X[:, :, 1:]
            X = Y & Cw
        out.append(((kw, kh), list(zip(xs.tolist(), ys.tolist())), X))
    return out


def placement_matrix(g, defs, weights=None):
    """-> (scipy csr R [placements x h*w] of the reach sets, costs int64[placements]) over every in-bounds placement"""
    h, w = g.shape
    rows, cols, costs, n = [], [], [], 0
    for (kw, kh), anchors, X in window_reach(g, defs):
        p, r, c = np.nonzero(X)
        xs = np.array([a[0] for a in anchors])[p] - HALO + c
        ys = np.array([a[1] for a in anchors])[p] - HALO + r
        rows.append(p + n)
        cols.append(ys * w + xs)
        costs += [1 if weights is None else _platform_cost(kw, kh, weights)] * len(anchors)
        n += len(anchors)
    R = scipy.sparse.csr_matrix((np.ones(sum(len(x) for x in rows), np.int64), (np.concatenate(rows), np.concatenate(cols))), shape=(n, h * w))
    return R, np.array(costs, np.int64)


def certificate(g, defs, weights, wts):
    """-> (total, max load, bound) recomputed exactly from integer weights"""
    R, cost = placement_matrix(g, defs, weights)
    k = np.asarray(wts, np.int64).reshape(-1)
    loads = R @ k
    total = int(k.sum())
    carrying = np.flatnonzero(loads > 0)
    if len(carrying) == 0:
        return total, 0, 0
    return total, int(loads.max()), math.ceil(min(Fraction(total * int(cost[i]), int(loads[i])) for i in carrying))


def reference_lp(g, defs, weights=None):
    """HiGHS on the same LP: max sum y over ceiling tiles, R y <= cost (placements that cost nothing fix their reach at 0)"""
    R, cost = placement_matrix(g, defs, weights)
    cols = np.flatnonzero(g.reshape(-1))
    A = R[:, cols]
    keep = np.asarray(A.sum(1)).reshape(-1) > 0
    res = scipy.optimize.linprog(-np.ones(len(cols)), A_ub=A[keep], b_ub=cost[keep].astype(float), bounds=(0, None), method="highs")
    assert res.status == 0, res.message
    return -res.fun


def c4():
    return synth_terrain(256, 256, seed=1, t=0)


def dense96x72():
    return synth_terrain(96, 72, seed=4, t=1, density_q24=int(0.85 * (1 << 24)))


# ---------------------------------------------------------------------------------------------------------- CPU tests
def test_window_reach_matches_full_grid_reach_sets():
    """The windowed reach of the reference is validate()'s rule (test_lp_reference.reach_sets, itself checked against the oracle)."""
    rng = np.random.default_rng(5)
    for g, defs in ((synth_terrain(13, 11, seed=3, t=0), DEFS_DEFAULT), ((rng.random((9, 14)) < 0.8).astype(np.uint8), [(1, 1), (1, 3), (3, 3)]),
                    (np.ones((1, 20), np.uint8), DEFS_1X1)):
        full, where = reach_sets(g, defs)
        R, _ = placement_matrix(g, defs)
        assert R.shape[0] == len(where)
        assert np.array_equal(R.toarray().astype(bool), full.reshape(len(where), -1))


# ---------------------------------------------------------------------------------------------------------- GPU tests
@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def _api(defs, weights):
    return [T.PlatformDef(*d) for d in defs], None if weights is None else {T.PlatformDef(*d): v for d, v in weights.items()}


def _bound(eng, g, defs, weights=None, **kw):
    d, w = _api(defs, weights)
    return eng.lower_bound_lp(T.WorldGrid(g), d, weights=w, **kw)


def _check(g, defs, weights, r):
    wts = r["weights"].astype(np.int64)
    assert wts.shape == g.shape and (wts >= 0).all() and not wts[g == 0].any()
    total, max_load, bound = certificate(g, defs, weights, wts)
    assert (r["total"], r["max_load"], r["bound"]) == (total, max_load, bound)
    assert not r["optimal"]


def _isolated():
    g = np.zeros((40, 40), np.uint8)
    g[::9, ::9] = 1
    return g


SHAPES = {"33x33": lambda: synth_terrain(33, 33, seed=2, t=0), "40x36": lambda: synth_terrain(40, 36, seed=3, t=1),
          "64x64": lambda: synth_terrain(64, 64, seed=1, t=0), "256x40": lambda: synth_terrain(256, 40, seed=5, t=0),
          "corridor1x256": lambda: np.ones((1, 256), np.uint8), "zero40x40": lambda: np.zeros((40, 40), np.uint8), "isolated": _isolated}
EXACT = [(s, "1x1") for s in SHAPES] + [("33x33", "default8"), ("40x36", "gui"), ("64x64", "default8"), ("isolated", "gui")]
PSETS = {"1x1": (DEFS_1X1, None), "default8": (DEFS_DEFAULT, None), "gui": (DEFS_DEFAULT, GUI_WEIGHTS)}


@pytest.mark.gpu
@pytest.mark.parametrize("shape,pset", EXACT, ids=[f"{s}/{p}" for s, p in EXACT])
def test_certificate_is_exact(eng, shape, pset):
    """total, max load and bound are what the reported integer weights give over every in-bounds placement."""
    g = SHAPES[shape]()
    defs, weights = PSETS[pset]
    r = _bound(eng, g, defs, weights, max_pivots=600)
    _check(g, defs, weights, r)
    if not g.any():
        assert r["bound"] == 0 and r["total"] == 0 and r["pivots"] == 0
    if shape == "isolated" and pset == "1x1":
        assert r["bound"] == int(g.sum())          # no placement reaches two of the tiles: every tile needs its own platform


QUALITY = [(n, p) for n in (48, 64) for p in ("1x1", "default8", "gui")]


@pytest.mark.gpu
@pytest.mark.parametrize("n,pset", QUALITY, ids=[f"{n}x{n}/{p}" for n, p in QUALITY])
def test_bound_reaches_98_percent_of_the_lp(eng, n, pset):
    g = synth_terrain(n, n, seed=1, t=0)
    defs, weights = PSETS[pset]
    lp = reference_lp(g, defs, weights)
    r = _bound(eng, g, defs, weights)
    _check(g, defs, weights, r)
    print(f"{n}x{n} {pset}: certified {r['bound']} / LP {lp:.3f} = {r['bound'] / lp:.4f} after {r['pivots']} iterations")
    assert r["bound"] <= math.ceil(lp - 1e-6)
    assert r["bound"] >= 0.98 * lp


def _layout_cost(layout, weights):
    if weights is None:
        return layout.platform_count()
    return sum(_platform_cost(p.definition.width, p.definition.height, weights) for p in layout.platforms().values())


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True], ids=["count", "gui"])
def test_bound_below_window_placement_search(eng, weighted):
    g = dense96x72()
    weights = GUI_WEIGHTS if weighted else None
    d, w = _api(DEFS_DEFAULT, weights)
    s = eng.search(T.WorldGrid(g), d, seed=1, kernel=T.KERNEL_WINDOW_PLACEMENTS)
    if w:
        s.set_weights(w)
    for _ in range(4):
        s.run(2000, 0)
    lay = s.best_layout()
    s.close()
    plats = [(p.x, p.y, p.definition.width, p.definition.height, int(p.rotated)) for p in lay.platforms().values()]
    assert O.validate(g, plats).is_valid
    r = _bound(eng, g, DEFS_DEFAULT, weights)
    print(f"dense 96x72 {'GUI weights' if weighted else 'count'}: bound {r['bound']} <= search {_layout_cost(lay, weights)}")
    assert 0 < r["bound"] <= _layout_cost(lay, weights)


def c4_lp():
    """HiGHS (interior point) on C4 with 1x1 supports, R built sparsely: ((I + A)^3 > 0) over the ceiling's 4-neighbour adjacency"""
    g = c4()
    h, w = g.shape
    idx = -np.ones(g.shape, np.int64)
    cols = np.flatnonzero(g.reshape(-1))
    idx.reshape(-1)[cols] = np.arange(len(cols))
    src, dst = [], []
    for dy, dx in ((0, 1), (1, 0)):
        a, b = idx[:h - dy, :w - dx], idx[dy:, dx:]
        m = (a >= 0) & (b >= 0)
        src += [a[m], b[m]]
        dst += [b[m], a[m]]
    n = len(cols)
    A = scipy.sparse.csr_matrix((np.ones(sum(len(x) for x in src)), (np.concatenate(src), np.concatenate(dst))), shape=(n, n))
    M = A + scipy.sparse.identity(n, format="csr")
    R = ((M @ M @ M) > 0).astype(np.float64)
    res = scipy.optimize.linprog(-np.ones(n), A_ub=R, b_ub=np.ones(n), bounds=(0, None), method="highs-ipm")
    assert res.status == 0, res.message
    return -res.fun


@pytest.mark.gpu
def test_c4_bound_beats_packing_and_reaches_99_percent(eng):
    g = c4()
    grid = T.WorldGrid(g)
    packing = len(eng.lower_bound(grid, seed=1))
    r = eng.lower_bound_lp(grid)
    lp = c4_lp()
    print(f"C4 1x1: packing {packing}, certified {r['bound']} / LP {lp:.3f} = {r['bound'] / lp:.4f} after {r['pivots']} iterations, "
          f"{eng.stats()['device_ms']:.1f} ms")
    assert abs(lp - 4165.017) < 0.01
    assert r["bound"] > packing and r["bound"] >= 0.99 * lp and r["bound"] <= math.ceil(lp)
    s = eng.search(grid, seed=1)
    for _ in range(2):
        s.run(2000, 0)
    count = s.best_layout().platform_count()
    s.close()
    assert r["bound"] <= count


@pytest.mark.gpu
def test_repeat_target_and_cap(eng):
    """Two calls give identical weights; a target the full run reaches is reached by the early stop; a cap only weakens the bound."""
    g = SHAPES["64x64"]()
    full = _bound(eng, g, DEFS_DEFAULT, GUI_WEIGHTS)
    again = _bound(eng, g, DEFS_DEFAULT, GUI_WEIGHTS)
    assert np.array_equal(full["weights"], again["weights"]) and full["bound"] == again["bound"] and full["pivots"] == again["pivots"]
    for t in (1, full["bound"] // 2, full["bound"]):
        r = _bound(eng, g, DEFS_DEFAULT, GUI_WEIGHTS, target=t)
        _check(g, DEFS_DEFAULT, GUI_WEIGHTS, r)
        assert r["bound"] >= t and r["pivots"] <= full["pivots"]
    early = _bound(eng, g, DEFS_DEFAULT, GUI_WEIGHTS, target=1)
    assert early["pivots"] < full["pivots"]
    for cap in (1, 50, 300):
        r = _bound(eng, g, DEFS_DEFAULT, GUI_WEIGHTS, max_pivots=cap)
        _check(g, DEFS_DEFAULT, GUI_WEIGHTS, r)
        assert r["pivots"] == cap and r["bound"] <= full["bound"]


@pytest.mark.gpu
def test_unsupported_inputs(eng):
    with pytest.raises(T.TssError, match="256x256"):
        eng.lower_bound_lp(T.WorldGrid(np.ones((257, 257), np.uint8)))
    g = T.WorldGrid(np.ones((40, 40), np.uint8))
    with pytest.raises(T.TssError, match="6x6"):
        eng.lower_bound_lp(g, [T.PlatformDef(1, 1), T.PlatformDef(7, 7)])
    seventeen = [(1, 1)] + [(1, k) for k in range(2, 7)] + [(2, 3), (2, 4), (2, 5)]
    assert len(_key_dims(seventeen)) == 17
    with pytest.raises(T.TssError, match="dims keys"):
        eng.lower_bound_lp(g, [T.PlatformDef(*d) for d in seventeen])
    sixteen = seventeen[:-1] + [(2, 2)]
    assert len(_key_dims(sixteen)) == 16
    r = eng.lower_bound_lp(g, [T.PlatformDef(*d) for d in sixteen], max_pivots=100)
    _check(np.ones((40, 40), np.uint8), sixteen, None, r)
