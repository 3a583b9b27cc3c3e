"""Parity tests proper: the CUDA path (through the C ABI of libtss) against the oracle on the same seeded inputs,
against the committed golden fixtures, and through size-independent properties at BASELINE.json's full sizes.
Bit-exact everywhere: the path is integer / boolean only (SURVEY.md §8: no floating point)."""
import os

import numpy as np
import pytest

import oracle.oracle as O
import timberborn_support_solver_b200 as T
from conftest import golden, rows_to_grid, synth_terrain

pytestmark = pytest.mark.gpu
ONE = T.PlatformDef(1, 1)


@pytest.fixture(scope="module")
def eng():
    e = T.Engine(0)
    yield e
    e.close()


def tup(p):
    return (p.x, p.y, p.definition.width, p.definition.height, int(p.rotated))


def random_sites(rng, n, h, w, p):
    return (rng.random((n, h, w)) < p).astype(np.uint8)


def pack_rows(mask):
    """uint8[..., h, w] -> uint32[..., h, ceil(w/32)] (tss.h bit-packed rows)"""
    h, w = mask.shape[-2:]
    wpr = (w + 31) // 32
    pad = np.zeros(mask.shape[:-1] + (wpr * 32,), np.uint8)
    pad[..., :w] = mask
    bits = pad.reshape(mask.shape[:-1] + (wpr, 32)).astype(np.uint64)
    return (bits << np.arange(32, dtype=np.uint64)).sum(-1).astype(np.uint32)


# =============================================================================== kernel (a): coverage evaluator
@pytest.mark.parametrize("w,h", [(1, 1), (5, 6), (8, 8), (7, 3), (16, 16), (11, 7), (13, 29), (21, 16), (32, 32), (32, 5), (17, 32)])
def test_eval_sites_small_grids_match_validate(eng, w, h):
    rng = np.random.default_rng(w * 100 + h)
    for density in (1.0, 0.7, 0.3):
        grid = (rng.random((h, w)) < density).astype(np.uint8)
        sites = random_sites(rng, 257, h, w, 0.08)
        sites[0] = 0                 # empty layout: everything unsupported
        sites[1] = 1                 # a support everywhere
        unc, cnt = eng.eval_sites(T.WorldGrid(grid), sites)
        o_unc, o_cnt, _ = O.validate_sites_batch(grid, sites)
        assert np.array_equal(unc, o_unc) and np.array_equal(cnt, o_cnt), (w, h, density)
        assert unc[0] == grid.sum() and unc[1] == 0


def test_eval_packed_equals_eval_sites(eng, fixtures):
    rng = np.random.default_rng(3)
    for name in ("ex1", "ex2", "ex3"):
        g = fixtures[name]
        h, w = g.shape
        sites = random_sites(rng, 100, h, w, 0.1)
        unc, cnt = eng.eval_sites(T.WorldGrid(g), sites)
        unc2, cnt2 = eng.eval_packed(pack_rows(g), w, h, pack_rows(sites))
        assert np.array_equal(unc, unc2) and np.array_equal(cnt, cnt2)


@pytest.mark.parametrize("w,h", [(40, 40), (33, 7), (64, 64), (100, 37), (256, 256)])
def test_eval_sites_tiled_grids_match_validate(eng, w, h):
    rng = np.random.default_rng(w + h)
    grid = synth_terrain(w, h, seed=1)
    n = 6 if w * h > 10000 else 40
    sites = random_sites(rng, n, h, w, 0.05)
    unc, cnt = eng.eval_sites(T.WorldGrid(grid), sites)
    o_unc, o_cnt, _ = O.validate_sites_batch(grid, sites)
    assert np.array_equal(unc, o_unc) and np.array_equal(cnt, o_cnt)


def test_readme_golden_layouts_validate_on_gpu(eng, readme):
    grid, layouts = readme
    sites = np.zeros((len(layouts), 16, 21), np.uint8)
    for i, lay in enumerate(layouts):
        for x, y in lay["supports"]:
            sites[i, y, x] = 1
    unc, cnt = eng.eval_sites(T.WorldGrid(grid), sites)
    assert unc.tolist() == [0, 0, 0, 0] and cnt.tolist() == [18, 17, 16, 15]      # README.md:47-116
    for lay in layouts:
        v = T.PlatformLayout(T.Platform(x, y, ONE) for x, y in lay["supports"]).validate(T.World(T.WorldGrid(grid)), eng)
        assert v.is_valid()


def test_geodesic_not_manhattan(eng):
    g = T.WorldGrid(rows_to_grid(["XXX XXX"]))
    v = eng.validate(g, [T.Platform(0, 0, ONE)])
    assert v.unsupported_terrain == {(4, 0), (5, 0), (6, 0)}
    g = T.WorldGrid(rows_to_grid(["XXXXXXX"]))
    assert eng.validate(g, [T.Platform(3, 0, ONE)]).is_valid() and not eng.validate(g, [T.Platform(2, 0, ONE)]).is_valid()


def random_platforms(rng, w, h, n):
    defs = [(1, 1), (1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (3, 3), (5, 5)]
    out = []
    for _ in range(n):
        d = defs[rng.integers(len(defs))]
        out.append((int(rng.integers(-2, w + 1)), int(rng.integers(-2, h + 1)), d[0], d[1], int(rng.integers(2))))
    return list({(p[0], p[1]): p for p in out}.values())  # one platform per anchor, like the reference's HashMap


@pytest.mark.parametrize("w,h", [(5, 6), (21, 16), (32, 32), (50, 20), (256, 256)])
def test_validate_platform_layouts_match_oracle(eng, w, h):
    rng = np.random.default_rng(w * 7 + h)
    grid = synth_terrain(w, h, seed=2, density_q24=int(0.8 * (1 << 24)))
    layouts = [random_platforms(rng, w, h, int(rng.integers(0, max(2, w * h // 30)))) for _ in range(8 if w * h < 5000 else 2)]
    out = eng.eval_platforms(T.WorldGrid(grid), [[T.Platform(p[0], p[1], T.PlatformDef(p[2], p[3]), bool(p[4])) for p in l] for l in layouts])
    for i, l in enumerate(layouts):
        ref = O.validate(grid, l)
        assert out[i].tolist() == [int(ref.unsupported.sum()), len(l), len(ref.overlapping), len(ref.out_of_bounds)], (w, h, i)
        v = eng.validate(T.WorldGrid(grid), [T.Platform(p[0], p[1], T.PlatformDef(p[2], p[3]), bool(p[4])) for p in l])
        assert {(x, y) for y, x in zip(*np.nonzero(ref.unsupported))} == v.unsupported_terrain
        assert {tup(p) for p in v.overlapping_platforms} == set(ref.overlapping)
        assert {tup(p) for p in v.out_of_bounds_platforms} == set(ref.out_of_bounds)


def test_eval_full_size_properties(eng):
    """C4 / C5 sizes: properties instead of the (slow) oracle — monotone in the support set, exact on the extremes,
    and one random 256x256 layout cross-checked against the oracle."""
    rng = np.random.default_rng(0)
    grid = synth_terrain(256, 256, seed=1)
    n_ceiling = int(grid.sum())
    assert 0.69 * 65536 < n_ceiling < 0.71 * 65536                        # density 0.7 (SURVEY.md §8d generator)
    a = random_sites(rng, 3, 256, 256, 0.03)
    b = a | random_sites(rng, 3, 256, 256, 0.03)
    ua, _ = eng.eval_sites(T.WorldGrid(grid), a)
    ub, cb = eng.eval_sites(T.WorldGrid(grid), b)
    assert (ub <= ua).all() and (cb == b.reshape(3, -1).sum(1)).all()
    u, _ = eng.eval_sites(T.WorldGrid(grid), np.stack([np.zeros_like(grid), grid]))
    assert u.tolist() == [n_ceiling, 0]
    o_unc, _, _ = O.validate_sites_batch(grid, a[:1])
    assert o_unc[0] == ua[0]
    # 4096 terrains of the C5 generator, supports on a 5-lattice: evaluated per terrain == oracle on a sample
    terr = np.stack([synth_terrain(32, 32, seed=1, t=t) for t in range(64)])
    lat = np.zeros((32, 32), np.uint8)
    lat[2::5, 2::5] = 1
    for t in (0, 17, 63):
        u, c = eng.eval_sites(T.WorldGrid(terr[t]), lat[None])
        o_u, o_c, _ = O.validate_sites_batch(terr[t], lat[None])
        assert u[0] == o_u[0] and c[0] == o_c[0] == 36


# =============================================================================== kernel (c): CNF check / propagate
@pytest.mark.parametrize("name,defs", [("ex1", "1x1"), ("ex3", "1x1"), ("ex1", "default"), ("ex3", "default")])
def test_cnf_check_matches_oracle(eng, fixtures, name, defs):
    d = T.PLATFORMS_DEFAULT[:1] if defs == "1x1" else T.PLATFORMS_DEFAULT
    g = fixtures[name]
    enc = T.Encoding.encode(d, T.WorldGrid(g))
    cnf = enc.with_limits(T.PlatformLimits.new_unweighted({ONE: 5}))
    ocnf = O.Encoding([x.dims() for x in d], g).with_limits({(1, 1): 5})
    dev = eng.upload_cnf(cnf)
    rng = np.random.default_rng(11)
    a = rng.integers(0, 3, (70, cnf.n_vars + 1)).astype(np.uint8)   # False / True / DontCare
    a[0] = 1
    a[1] = 0
    r, model, _ = ocnf.solve()
    assert r == 10
    a[2] = model
    nf, first = dev.check(a)
    for i in range(len(a)):
        want = ocnf.count_falsified(a[i])
        assert (int(nf[i]), int(first[i])) == want, i
    assert nf[2] == 0 and first[2] == -1


def _plat_only_assignment(enc, cnf, supports):
    """platform variables decided (the given 1x1 supports True, every other tile False), terrain-layer and cardinality
    variables open: what unit propagation has to complete (src/encoder.rs:500-544)"""
    a = np.full(cnf.n_vars + 1, 2, np.uint8)
    pv = enc.vars().plat_var[:, 0]
    a[pv] = 0
    w = enc.vars().width
    for x, y in supports:
        a[pv[y * w + x]] = 1
    return a


def _check_propagation(eng, g, enc, cnf, ocnf, batch, layouts, bound):
    """kernel (c) propagation == the oracle's (oracle/capi.cpp tsso_cnf_propagate): full assignment, conflict verdict and
    the number of synchronous rounds; and SURVEY.md §7 step 1: validate(layout) and count <= bound <=> no conflict."""
    dev = eng.upload_cnf(cnf)
    out, conflict, rounds = dev.propagate(np.stack(batch))
    want_rounds, n_clean = 0, 0
    for i, a in enumerate(batch):
        want, wc, wr = ocnf.propagate(a)
        want_rounds = max(want_rounds, wr)
        assert np.array_equal(out[i][1:], want[1:]), i          # the whole propagated assignment, conflict or not
        assert (conflict[i] >= 0) == (wc >= 0), i
        if wc >= 0:                                              # the reported clause is falsified at the fixpoint (any such clause is a valid witness)
            cl = cnf.clauses()[int(conflict[i])]
            assert all(out[i][abs(l)] == (0 if l > 0 else 1) for l in cl), i
        else:
            n_clean += 1
        plats = [(x, y, 1, 1, 0) for x, y in layouts[i]]
        ok = O.validate(g, plats).is_valid and len(plats) <= bound
        assert ok == (conflict[i] < 0), i
    assert rounds == want_rounds
    return n_clean


def test_cnf_propagate_matches_oracle_random(eng, fixtures):
    g = fixtures["ex1"]
    h, w = g.shape
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT[:1], T.WorldGrid(g))
    cnf = enc.with_limits(T.PlatformLimits.new_unweighted({ONE: 3}))
    ocnf = O.Encoding(O.PLATFORMS_1X1, g).with_limits({(1, 1): 3})
    assert cnf.clauses() == ocnf.clauses()
    rng = np.random.default_rng(2)
    batch, layouts = [], []
    for i in range(40):
        k = int(rng.integers(0, 5))
        tiles = rng.choice(w * h, k, replace=False)
        layouts.append([(int(t % w), int(t // w)) for t in tiles])
        batch.append(_plat_only_assignment(enc, cnf, layouts[-1]))
    # valid layouts too (the conflict-free side): every 3-support layout the exhaustive search finds on this 30-tile terrain
    import itertools
    ceil = [(x, y) for y in range(h) for x in range(w) if g[y, x]]
    for combo in itertools.combinations(ceil, 3):
        if len(batch) >= 40 + 24:
            break
        if O.validate(g, [(x, y, 1, 1, 0) for x, y in combo]).is_valid:
            layouts.append(list(combo))
            batch.append(_plat_only_assignment(enc, cnf, combo))
    n_clean = _check_propagation(eng, g, enc, cnf, ocnf, batch, layouts, 3)
    assert n_clean >= 10


def test_cnf_propagate_on_optimum_witnesses(eng, fixtures, readme):
    """The conflict-free side on real witnesses: the survey's three optimum layouts, the four README layouts and fresh SLS
    witnesses, with ONLY the platform variables fixed — propagation has to derive every terrain layer and every totalizer
    variable of the at-most-n bound; the result must equal the oracle's propagation variable for variable."""
    terrains = {"rect16": np.ones((16, 16), np.uint8), "ex2": fixtures["ex2"], "readme": readme[0]}
    cases = [(w["terrain"], [tuple(p) for p in w["supports"]], w["optimum"]) for w in golden("survey_witnesses")["witnesses"]]
    cases += [("readme", [tuple(p) for p in lay["supports"]], len(lay["supports"])) for lay in readme[1]]
    for name, opt in (("rect16", 15), ("readme", 14), ("ex2", 14)):
        res, lay = eng.solve_upper_bound(T.WorldGrid(terrains[name]), card_limit=opt, seed=5, max_steps=200000)
        assert res == T.SAT
        cases.append((name, [(p.x, p.y) for p in lay.platforms().values()], opt))
    n_clean = 0
    for name, sup, bound in cases:
        g = terrains[name]
        enc = T.Encoding.encode(T.PLATFORMS_DEFAULT[:1], T.WorldGrid(g))
        cnf = enc.with_limits(T.PlatformLimits.new_unweighted({ONE: bound}))
        ocnf = O.Encoding(O.PLATFORMS_1X1, g).with_limits({(1, 1): bound})
        assert cnf.clauses() == ocnf.clauses()
        # the witness itself, the witness with one support dropped (coverage conflict), and against a bound one too small
        batch = [_plat_only_assignment(enc, cnf, sup), _plat_only_assignment(enc, cnf, sup[1:])]
        n_clean += _check_propagation(eng, g, enc, cnf, ocnf, batch, [sup, sup[1:]], bound)
        # propagation alone leaves the terrain layers of covered tiles open (T_l -> OR of T_l+1 is not unit); the model the exact
        # solver is handed takes them from the evaluator's support layers (tss_layout_to_assignment), then propagation fills
        # in the totalizer: the recipe of api.GpuBoundSolver.solve and of the Rust shim (INTEGRATION.md)
        lay = T.PlatformLayout(T.Platform(x, y, ONE, False) for x, y in sup)
        full = np.full((1, cnf.n_vars + 1), 2, np.uint8)
        base = eng.layout_to_assignment(enc, lay)
        full[0, : len(base)] = base
        prop, conflict, _ = eng.upload_cnf(cnf).propagate(full)
        want, wc, _ = ocnf.propagate(full[0])
        assert conflict[0] < 0 and wc < 0 and np.array_equal(prop[0][1:], want[1:])
        prop[prop == 2] = 0
        assert ocnf.count_falsified(prop[0]) == (0, -1)
        # the same completion in ONE launch (tss_witness_for_cnf -> cnf_complete_kernel: in-place propagation, open variables
        # False, every clause checked): the same model, variable for variable; not a model when a support is missing
        dev = eng.upload_cnf(cnf)
        fused = dev.witness(enc, lay)
        assert fused is not None and np.array_equal(fused[1:], prop[0][1:])
        assert dev.witness(enc, T.PlatformLayout(T.Platform(x, y, ONE, False) for x, y in sup[1:])) is None
        tight = enc.with_limits(T.PlatformLimits.new_unweighted({ONE: bound - 1}))
        otight = O.Encoding(O.PLATFORMS_1X1, g).with_limits({(1, 1): bound - 1})
        assert _check_propagation(eng, g, enc, tight, otight, [_plat_only_assignment(enc, tight, sup)], [sup], bound - 1) == 0
        assert eng.upload_cnf(tight).witness(enc, lay) is None          # one platform more than the bound allows: a conflict in the totalizer
    assert n_clean == len(cases) >= 10


def _random_cnf(rng, n_vars, n_clauses, chain, hidden):
    """Random clause set with unit-propagation structure: `chain` implication chains x -> y -> z ..., random clauses of 1..9
    literals, a few long ones.  With `hidden` (a full assignment) every clause is made true under it — propagation from any part
    of it can then never conflict; without, literals are random and an empty clause may appear."""
    clauses = []
    order = rng.permutation(n_vars) + 1
    for i in range(chain):
        a, b = int(order[i % n_vars]), int(order[(i + 1) % n_vars])
        clauses.append((-a if rng.random() < 0.8 else a, b if rng.random() < 0.8 else -b))
    for _ in range(n_clauses):
        k = int(rng.choice([1, 2, 2, 3, 3, 3, 4, 5, 6, 9]))
        vs = rng.choice(n_vars, size=min(k, n_vars), replace=False) + 1
        clauses.append(tuple(int(v) if rng.random() < 0.5 else -int(v) for v in vs))
    if hidden is not None:
        fixed = []
        for c in clauses:
            if not any(hidden[abs(l)] == (1 if l > 0 else 0) for l in c):
                j = int(rng.integers(len(c)))
                c = c[:j] + (-c[j],) + c[j + 1:]
            fixed.append(c)
        clauses = fixed
    elif rng.random() < 0.2:
        clauses.append(())
    perm = rng.permutation(len(clauses))
    clauses = [clauses[i] for i in perm]
    lits = np.array([l for c in clauses for l in c], np.int32)
    offs = np.zeros(len(clauses) + 1, np.uint32)
    offs[1:] = np.cumsum([len(c) for c in clauses])
    return clauses, lits, offs


@pytest.mark.parametrize("n_vars,n_clauses,cases", [(12, 20, 60), (300, 500, 40), (5000, 12000, 12), (40000, 60000, 4), (230000, 100000, 2)])
def test_cnf_complete_random_clause_sets_match_oracle(eng, n_vars, n_clauses, cases):
    """tss_cnf_complete (one fused launch, in-place propagation; 16-bit resident clauses below 32 768 variables, the int4 copy
    above, the batch kernels beyond one CTA's shared memory) on clause sets no encoder produces — chains, long and empty clauses,
    conflicts — against the oracle's synchronous unit propagation: same conflict verdict; without a conflict the same completed
    assignment, variable for variable, and the same number of falsified clauses."""
    rng = np.random.default_rng(n_vars)
    n_conflict = n_clean = 0
    for case in range(cases):
        hidden = rng.integers(0, 2, n_vars + 1).astype(np.uint8) if case % 2 == 0 else None
        clauses, lits, offs = _random_cnf(rng, n_vars, n_clauses, chain=n_vars // 2, hidden=hidden)
        a = np.full(n_vars + 1, 2, np.uint8)
        decided = rng.random(n_vars + 1) < rng.choice([0.0, 0.05, 0.3, 0.6])
        a[decided] = hidden[decided] if hidden is not None else rng.integers(0, 2, int(decided.sum()))
        a[0] = 2
        want, wc, _ = O.propagate_csr(lits, offs, n_vars, a)
        dev = eng.upload_cnf(T.Cnf(n_vars, lits, offs))
        got, conflict, nf = dev.complete(a)
        assert (conflict >= 0) == (wc >= 0), (case, conflict, wc)
        if wc >= 0:
            n_conflict += 1
            cl = clauses[conflict]                       # the reported clause has no true and no open literal in the returned state
            assert all(got[abs(l)] == (0 if l > 0 else 1) for l in cl), case
            continue
        n_clean += 1
        want[want == 2] = 0
        assert np.array_equal(got[1:], want[1:]), case
        bad = sum(1 for c in clauses if not any(want[abs(l)] == (1 if l > 0 else 0) for l in c)) if n_vars <= 5000 else None
        if bad is not None:
            assert nf == bad, (case, nf, bad)
        else:                                            # large sets: the batch check kernel is the yardstick (itself tested against the oracle above)
            assert nf == dev.check(want[None, :])[0][0], case
    assert n_clean >= cases // 2 and n_conflict > 0


# =============================================================================== kernel (b): batched SLS
KNOWN_OPTIMA = [("ex1", 3), ("ex3", 4), ("ex2", 14)]   # proven by the oracle's CDCL loop (tests/test_oracle.py) / SURVEY.md §6


@pytest.mark.parametrize("name,optimum", KNOWN_OPTIMA)
def test_sls_reaches_proven_optimum(eng, fixtures, name, optimum):
    g = T.WorldGrid(fixtures[name])
    res, layout = eng.solve_upper_bound(g, T.PLATFORMS_DEFAULT[:1], card_limit=optimum, seed=7, max_steps=200000)
    assert res == T.SAT and layout.platform_count() == optimum
    plats = [tup(p) for p in layout.platforms().values()]
    assert O.validate(g.data, plats).is_valid                                    # the reference's coverage check
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT[:1], g)
    a = eng.layout_to_assignment(enc, layout)
    ocnf = O.Encoding(O.PLATFORMS_1X1, g.data).cnf()
    assert ocnf.count_falsified(a) == (0, -1)                                    # the reference encoder's CNF
    assert eng.upload_cnf(enc.cnf()).check(a[None])[0][0] == 0                   # same, on the GPU (kernel c)
    # one below the proven optimum nothing is ever reported (the GPU proves nothing, it just must not lie)
    res, layout = eng.solve_upper_bound(g, T.PLATFORMS_DEFAULT[:1], card_limit=optimum - 1, seed=7, max_steps=3000)
    assert res == T.INTERRUPTED and layout is None


def test_sls_rect16_and_readme_terrain(eng, readme):
    optima = {k: v["optimum"] for k, v in golden("proofs").items()}      # proven by tests/golden/make_proofs.py (oracle CDCL and z3)
    for grid, key in ((np.ones((16, 16), np.uint8), "rect16/1x1"), (readme[0], "readme/1x1")):
        opt = optima[key]
        g = T.WorldGrid(grid)
        res, layout = eng.solve_upper_bound(g, card_limit=opt, seed=1, max_steps=200000)
        assert res == T.SAT and layout.platform_count() == opt                   # rect 16x16: 15; README terrain: 14, one better than its transcript reached
        plats = [tup(p) for p in layout.platforms().values()]
        assert O.validate(g.data, plats).is_valid                                # the reference's coverage check
        enc = T.Encoding.encode(T.PLATFORMS_DEFAULT[:1], g)
        a = eng.layout_to_assignment(enc, layout)
        assert O.Encoding(O.PLATFORMS_1X1, g.data).cnf().count_falsified(a) == (0, -1)   # the reference encoder's CNF
        assert eng.upload_cnf(enc.cnf()).check(a[None])[0][0] == 0               # same, on the GPU (kernel c)


TRAJECTORY_CASES = [((16, 16), 1), ((21, 16), 5), ((32, 32), 9), ((6, 5), 3), ((13, 29), 2), ((32, 16), 4), ((20, 17), 6), ((26, 16), 7), ((9, 12), 8)]


def _kernels_for(shape):
    w, h = shape
    ks = [T.KERNEL_WARP]
    if h <= 16:
        ks.append(T.KERNEL_HALF_WARP)
    if h <= 16 and w <= 26:
        ks.append(T.KERNEL_THREAD)
    return ks


@pytest.mark.parametrize("shape,seed,kernel", [(sh, sd, k) for sh, sd in TRAJECTORY_CASES for k in _kernels_for(sh)])
def test_sls_trajectories_bit_exact_vs_model(eng, fixtures, shape, seed, kernel):
    """The three kernels (one chain per warp; two chains per warp for grids of <= 16 rows; one chain per thread for grids
    of <= 16 rows x 26 columns) and the scalar CPU model (oracle/sls_model.cpp) execute the same published step rule with
    the same counter-based RNG: every chain's supports, best layout, counters and step count agree bit for bit across epochs."""
    w, h = shape
    grid = {(16, 16): np.ones((16, 16), np.uint8), (21, 16): fixtures["ex2"], (6, 5): fixtures["ex1"].T.copy()}.get(shape)
    if grid is None:
        grid = synth_terrain(w, h, seed=1, t=4)
    n_chains, offset = 23, 100      # odd: the last warp of the half-warp kernel runs a single chain
    if kernel == T.KERNEL_THREAD:
        n_chains = 150              # two CTAs, the second one partially filled
    epochs = [(50, 1 << 20, 0), (300, 1 << 20, 0), (1000, 1 << 20, 0)]
    s = eng.search(T.WorldGrid(grid), seed=seed, n_chains=n_chains, chain_offset=offset, kernel=kernel)
    flips0 = eng.stats()["sls_flips"]
    for steps, _, target in epochs:
        s.run(steps, target)
    got = s.read_chains()
    want = O.sls_model(grid, n_chains, epochs, seed=seed, chain_offset=offset, share_bound=True)
    # the flat-array CPU port (bench.py's CPU arm) replays the same trajectories and counts flips (supports added + removed,
    # the unit of the bench line): the kernels' device-wide flip counter must equal its sum over the chains
    flat = O.sls_flat(grid, n_chains, epochs, seed=seed, chain_offset=offset, share_bound=True, threads=2)
    assert all(np.array_equal(flat[key], want[key]) for key in ("S", "bestS", "k", "best", "step", "scored", "steps"))
    assert eng.stats()["sls_flips"] - flips0 == int(flat["flips"].sum())
    unpack = lambda rows: ((rows[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8)
    assert np.array_equal(got["k"], want["k"])
    assert np.array_equal(got["best"], want["best"])
    assert np.array_equal(got["step"], want["step"])
    assert np.array_equal(got["scored"], want["scored"])
    assert np.array_equal(unpack(got["S"]), want["S"])
    assert np.array_equal(unpack(got["bestS"]), want["bestS"])
    assert s.best_count() == int(want["best"].min())
    s.close()


def test_sls_long_epochs_split_at_32768_steps(eng):
    """A run longer than 32768 steps is executed as consecutive epochs (16-bit tabu stamps never wrap inside one): the
    thread-per-chain kernel (recent-removal ring instead of stamps) and the half-warp kernel still agree with the model."""
    grid = np.ones((8, 8), np.uint8)
    epochs = [(40000, 1 << 20, -1)]
    want = O.sls_model(grid, 40, epochs, seed=11, chain_offset=0, share_bound=True)
    for kernel in (T.KERNEL_HALF_WARP, T.KERNEL_THREAD):
        s = eng.search(T.WorldGrid(grid), seed=11, n_chains=40, kernel=kernel)
        s.run(40000, -1)
        got = s.read_chains()
        assert np.array_equal(got["k"], want["k"]) and np.array_equal(got["step"], want["step"]) and np.array_equal(got["scored"], want["scored"])
        assert np.array_equal(got["best"], want["best"])
        s.close()


@pytest.mark.parametrize("shape,kernel", [((16, 16), k) for k in (1, 2, 3)] + [((21, 16), k) for k in (2, 3)] + [((32, 32), 1)])
def test_sls_warm_start_dense_layouts_bit_exact(eng, fixtures, shape, kernel):
    """tss_search_write_chains: chains start from given layouts.  Dense starts (every tile / every other tile a support)
    drive the cover counts up to 25 per tile, i.e. through all five count planes (the thread kernel keeps the two high
    planes in global memory), and the chains then shed supports one by one: still bit-identical with the CPU model."""
    w, h = shape
    grid = {(16, 16): np.ones((16, 16), np.uint8), (21, 16): fixtures["ex2"]}.get(shape)
    if grid is None:
        grid = synth_terrain(w, h, seed=1, t=2)
    n_chains = 40 if kernel == T.KERNEL_THREAD else 10
    rng = np.random.default_rng(5)
    init = np.zeros((n_chains, 32, 32), np.uint8)
    for c in range(n_chains):
        dens = [1.0, 0.5, 0.25, 0.1][c % 4]
        init[c, :h, :w] = (rng.random((h, w)) < dens) & ((grid != 0) | (c % 8 >= 4))     # some chains also get supports under non-ceiling tiles
    rows = (init.astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(2, dtype=np.uint32)
    epochs = [(120, 1 << 20, -1), (200, 1 << 20, -1)]
    s = eng.search(T.WorldGrid(grid), seed=4, n_chains=n_chains, chain_offset=7, kernel=kernel)
    s.write_chains(rows)
    for steps, _, target in epochs:
        s.run(steps, target)
    got = s.read_chains()
    want = O.sls_model(grid, n_chains, epochs, seed=4, chain_offset=7, share_bound=True, init_S=init)
    unpack = lambda r: ((r[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8)
    for key in ("k", "best", "step", "scored"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(unpack(got["S"]), want["S"]) and np.array_equal(unpack(got["bestS"]), want["bestS"])
    s.close()
    with pytest.raises(T.TssError):   # supports outside the grid are rejected
        s2 = eng.search(T.WorldGrid(np.ones((5, 5), np.uint8)), n_chains=2)
        bad = np.zeros((2, 32), np.uint32)
        bad[1, 2] = 1 << 7
        s2.write_chains(bad)


@pytest.mark.parametrize("kernel", [1, 2, 3])
def test_sls_degenerate_terrains_match_model(eng, kernel):
    """No ceiling at all (the empty layout is complete at once, chains finish), a single tile, a one-row corridor, a
    terrain of isolated tiles (every tile needs its own support): every kernel variant agrees with the CPU model."""
    cases = [np.zeros((4, 7), np.uint8), np.pad(np.ones((1, 1), np.uint8), ((2, 3), (4, 1))), np.ones((1, 26), np.uint8),
             (np.indices((16, 16)).sum(0) % 2 == 0).astype(np.uint8) * (np.indices((16, 16))[0] % 2 == 0)]
    for grid in cases:
        grid = np.ascontiguousarray(grid, np.uint8)
        epochs = [(30, 1 << 20, 0), (200, 1 << 20, 0)]
        s = eng.search(T.WorldGrid(grid), seed=2, n_chains=33, chain_offset=3, kernel=kernel)
        for steps, _, target in epochs:
            s.run(steps, target)
        got = s.read_chains()
        want = O.sls_model(grid, 33, epochs, seed=2, chain_offset=3, share_bound=True)
        for key in ("k", "best", "step", "scored"):
            assert np.array_equal(got[key], want[key]), (key, grid.shape)
        unpack = lambda r: ((r[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8)
        assert np.array_equal(unpack(got["S"]), want["S"]) and np.array_equal(unpack(got["bestS"]), want["bestS"])
        best = s.best_count()
        assert best == int(want["best"].min()) and best == {0: 0, 1: 1, 26: 4}.get(int(grid.sum()), best)
        s.close()


@pytest.mark.parametrize("case", ["rect16", "ex2", "random26x16", "random12x9-dense"])
def test_sls_kernel_variants_agree_at_scale(eng, fixtures, case):
    """The CPU model is too slow for thousands of chains x tens of thousands of steps; at that scale the independent kernel
    implementations (thread per chain vs half-warp vs warp) are compared with each other instead: identical chain states,
    counters and bounds after every epoch, including an epoch longer than the 32768-step split."""
    grid = {"rect16": np.ones((16, 16), np.uint8), "ex2": fixtures["ex2"], "random26x16": synth_terrain(26, 16, seed=7, t=1),
            "random12x9-dense": synth_terrain(12, 9, seed=8, t=2, density_q24=int(0.93 * (1 << 24)))}[case]
    n_chains = 2048 + 77
    runs = {}
    for kernel in (T.KERNEL_THREAD, T.KERNEL_HALF_WARP, T.KERNEL_WARP):
        if kernel == T.KERNEL_WARP and case != "ex2":
            continue                                # (one three-way comparison is enough; the warp kernel is the slowest)
        s = eng.search(T.WorldGrid(grid), seed=21, n_chains=n_chains, chain_offset=5, kernel=kernel)
        snaps = []
        for steps in (700, 6000, 40000):
            s.run(steps, 0)
            snaps.append((s.best_count(), s.global_best()))
        st = s.read_chains()
        runs[kernel] = (snaps, st)
        s.close()
    ref_snaps, ref = runs[T.KERNEL_THREAD]
    for kernel, (snaps, st) in runs.items():
        assert snaps == ref_snaps, kernel
        for key in ("S", "bestS", "k", "best", "step", "scored"):
            assert np.array_equal(st[key], ref[key]), (kernel, key)


def test_fused_one_shot_launch_equals_the_epoch_by_epoch_path(fixtures):
    """tss_solve_upper_bound in latency mode runs its first epoch as ONE fused launch once the engine holds a workspace
    (rows as kernel parameters, per-CTA reach table, chains started in registers, last-CTA reduce + validation).  Same
    spec, same seeds: it returns exactly the layout of the first (unfused) call and of the persistent-portfolio API."""
    e = T.Engine(0)
    n_chains = e.device_info()["sm_count"] * 16
    second_epoch_needed = 0
    for grid, limit in ((np.ones((16, 16), np.uint8), 15), (fixtures["ex2"], 14), (fixtures["ex1"], 3)):
        g = T.WorldGrid(grid)
        for seed in ((11, 12) if limit != 14 else range(11, 23)):   # (ex2 at 14 sometimes needs more than the fused 32 steps)
            e2 = T.Engine(0)                                                     # no workspace yet: epoch-by-epoch path
            res_a, lay_a = e2.solve_upper_bound(g, card_limit=limit, seed=seed)
            launches_a = e2.stats()["kernel_launches"]
            res_b, lay_b = e2.solve_upper_bound(g, card_limit=limit, seed=seed)  # workspace cached: fused launch
            launches_b = e2.stats()["kernel_launches"] - launches_a
            e2.close()
            assert res_a == res_b == T.SAT and launches_b < launches_a
            pa, pb = sorted(lay_a.platforms()), sorted(lay_b.platforms())
            assert pa == pb and len(pa) <= limit
            s = e.search(g, seed=seed, n_chains=n_chains, kernel=T.KERNEL_HALF_WARP)
            s.set_bound(limit + 1)
            steps = 32
            while s.best_count() is None:
                s.run(steps, limit)
                steps *= 2
            assert sorted(s.best_layout().platforms()) == pa
            second_epoch_needed += steps > 64
            s.close()
    # the placement search (platform sets beyond {1x1}) has the same fused first epoch once a workspace of that set is cached
    for name, limit in (("ex1", 1), ("ex3", 1), ("ex2", 4)):
        g = T.WorldGrid(fixtures[name])
        for seed in (3, 4, 5):
            e2 = T.Engine(0)
            res_a, lay_a = e2.solve_upper_bound(g, T.PLATFORMS_DEFAULT, card_limit=limit, seed=seed)
            launches_a = e2.stats()["kernel_launches"]
            res_b, lay_b = e2.solve_upper_bound(g, T.PLATFORMS_DEFAULT, card_limit=limit, seed=seed)
            launches_b = e2.stats()["kernel_launches"] - launches_a
            res_c, lay_c = e2.solve_upper_bound(g, T.PLATFORMS_DEFAULT[:4], card_limit=None, seed=seed)   # another platform set: no fused launch, fresh keys
            e2.close()
            assert res_a == res_b == res_c == T.SAT and launches_b < launches_a
            assert sorted(lay_a.platforms().values()) == sorted(lay_b.platforms().values()) and lay_b.platform_count() <= limit
            assert O.validate(g.data, [tup(p) for p in lay_c.platforms().values()]).is_valid
            assert all(p.definition in T.PLATFORMS_DEFAULT[:4] for p in lay_c.platforms().values())
    # an infeasible bound with a give-up point: fused epoch, follow-up epochs, then UNKNOWN after exactly that many steps
    e2 = T.Engine(0)
    g = T.WorldGrid(np.ones((16, 16), np.uint8))
    e2.solve_upper_bound(g, card_limit=15, seed=1)
    res, lay = e2.solve_upper_bound(g, card_limit=14, seed=1, max_steps=-300)
    assert res == T.INTERRUPTED and lay is None and e2.stats()["last_solve_steps"] == 300
    res, lay = e2.solve_upper_bound(g, card_limit=15, seed=2)          # the workspace is intact afterwards
    assert res == T.SAT and lay.platform_count() == 15
    e2.close()
    e.close()


def test_kernel_variant_rejected_when_grid_does_not_fit(eng):
    with pytest.raises(T.TssError):
        eng.search(T.WorldGrid(np.ones((20, 20), np.uint8)), n_chains=8, kernel=T.KERNEL_THREAD)
    with pytest.raises(T.TssError):
        eng.search(T.WorldGrid(np.ones((16, 30), np.uint8).T.copy()), n_chains=8, kernel=T.KERNEL_HALF_WARP)   # 30 rows


def test_sls_bound_sharing_and_determinism(eng):
    g = T.WorldGrid(np.ones((16, 16)))
    runs = []
    for _ in range(2):
        s = eng.search(g, seed=3, n_chains=64)
        s.set_bound(17)                       # externally known bound (the all-reduce-min of a portfolio)
        s.run(400, 0)
        runs.append((s.best_count(), s.read_chains()))
        s.close()
    assert runs[0][0] == runs[1][0] and runs[0][0] is not None and runs[0][0] <= 16
    assert np.array_equal(runs[0][1]["S"], runs[1][1]["S"]) and np.array_equal(runs[0][1]["best"], runs[1][1]["best"])
    assert (runs[0][1]["best"][runs[0][1]["best"] < (1 << 20)] <= 16).all()       # nobody reports a layout >= the bound


@pytest.mark.parametrize("name,optimum", [("ex1", 1), ("ex3", 1), ("ex2", 4)])
def test_multi_platform_search_reaches_repl_optimum(eng, fixtures, name, optimum):
    """BASELINE.json configs[0]/[2]: the REPL solves with PLATFORMS_DEFAULT (crates/repl/src/main.rs:254); the proven optima
    (oracle CDCL loop, tests/test_oracle.py) are 1 / 1 / 4 platforms.  Witnesses pass the oracle's validate (coverage,
    overlap, bounds) and the reference encoder's full default-8 CNF."""
    g = T.WorldGrid(fixtures[name])
    res, layout = eng.solve_upper_bound(g, T.PLATFORMS_DEFAULT, card_limit=optimum, seed=5, max_steps=60000)
    assert res == T.SAT and layout.platform_count() == optimum
    plats = [tup(p) for p in layout.platforms().values()]
    assert O.validate(g.data, plats).is_valid
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, g)
    a = eng.layout_to_assignment(enc, layout)
    ref = O.Encoding(O.PLATFORMS_DEFAULT, g.data)
    assert ref.cnf().count_falsified(a) == (0, -1)
    assert sorted(ref.layout_from_assignment(a)) == sorted(plats)              # decode(encode(layout)) round trip
    assert eng.upload_cnf(enc.cnf()).check(a[None])[0][0] == 0
    res, layout = eng.solve_upper_bound(g, T.PLATFORMS_DEFAULT, card_limit=optimum - 1, seed=5, max_steps=2000)
    assert res == T.INTERRUPTED


def test_multi_platform_random_sets_match_exact_optimum(eng):
    """Small random terrains x platform sets: the GPU count equals the optimum proven by the oracle loop; layouts are
    valid (no overlap, in bounds, full coverage) under the oracle."""
    rng = np.random.default_rng(8)
    sets = [[(1, 1), (2, 2)], [(1, 1), (1, 3)], [(1, 1), (2, 3), (3, 3)], [(1, 1), (1, 2), (3, 3), (5, 5)]]
    for i in range(8):
        w, h = int(rng.integers(4, 10)), int(rng.integers(4, 10))
        grid = (rng.random((h, w)) < 0.8).astype(np.uint8)
        defs = sets[i % len(sets)]
        exact = O.solver_loop(grid, defs)
        assert exact["proved_optimal"]
        res, layout = eng.solve_upper_bound(T.WorldGrid(grid), [T.PlatformDef(*d) for d in defs], card_limit=len(exact["best"]), seed=i, max_steps=40000)
        assert res == T.SAT and layout.platform_count() == len(exact["best"]), (i, w, h, defs)
        assert O.validate(grid, [tup(p) for p in layout.platforms().values()]).is_valid


GUI_WEIGHTS = {(1, 1): 5, (1, 2): 1, (1, 3): 1, (1, 4): 1, (1, 5): 1, (1, 6): 1, (3, 3): 2, (5, 5): 4}   # crates/gui/src/app.rs:53-62


def oracle_min_weight(grid, defs, weights):
    """The GUI loop (crates/gui/src/app.rs:235-245) on the oracle: solve, weight = total_weight(layout), weight_limit =
    weight - 1, until the CDCL stand-in says UNSAT.  -> proven minimum total weight."""
    enc = O.Encoding(defs, grid)
    limit, best = None, None
    while True:
        r, a, _ = enc.with_limits(weights=weights, weight_limit=limit).solve()
        if r != 10:
            assert r == 20
            return best
        lay = O.trivial_optimization(grid, enc.layout_from_assignment(a))        # app.rs:157
        best = O.total_weight(lay, weights)
        if best <= 0:
            return best
        limit = best - 1


@pytest.mark.parametrize("case", ["ex1", "ex3", "ex2", "random-set", "weights"])
def test_placement_search_trajectories_bit_exact_vs_model(eng, fixtures, case):
    """The placement search (platform sets beyond {1x1}: what the REPL solves) against its scalar CPU model
    (oracle/slsm_model.cpp): every chain's placements in list order, best layout, objective value and step counter agree
    bit for bit across epochs, and so do the engine's candidate / step counters."""
    defs, weights = list(T.PLATFORMS_DEFAULT), None
    if case in ("ex1", "ex3", "ex2"):
        grid = fixtures[case]
    elif case == "random-set":
        grid = synth_terrain(20, 17, seed=3, t=1)
        defs = [T.PlatformDef(1, 1), T.PlatformDef(2, 3), T.PlatformDef(2, 2), T.PlatformDef(1, 4), T.PlatformDef(4, 4)]
    else:
        grid = synth_terrain(14, 12, seed=5, t=2, density_q24=int(0.85 * (1 << 24)))
        weights = {T.PlatformDef(1, 1): 3, T.PlatformDef(1, 3): 2, T.PlatformDef(3, 3): 4, T.PlatformDef(5, 5): 7}
    n_chains, offset, seed = 6, 50, 9
    epochs = [(40, 1 << 20, 0), (150, 1 << 20, 0), (400, 1 << 20, 0)]
    s = eng.search(T.WorldGrid(grid), defs, seed=seed, n_chains=n_chains, chain_offset=offset)
    if weights:
        s.set_weights(weights)
    st0 = eng.stats()
    for steps, _, target in epochs:
        s.run(steps, target)
    got = s.read_placements()
    st1 = eng.stats()
    key_dims = got["key_dims"]
    costs = [1] * len(key_dims)
    if weights:   # cost of a platform = sum of the weights of every def that fits inside its def (platform_layout.rs:174-183)
        canon = lambda w, h: (min(w, h), max(w, h))
        costs = [sum(v for d, v in weights.items() if canon(d.width, d.height)[0] <= canon(w, h)[0] and canon(d.width, d.height)[1] <= canon(w, h)[1])
                 for w, h in key_dims]
    want = O.slsm_model(grid, key_dims, costs, n_chains, epochs, seed=seed, chain_offset=offset, share_bound=True)
    for key in ("k", "best", "best_k", "step"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(got["items"], want["items"]) and np.array_equal(got["best_items"], want["best_items"])
    assert st1["candidates_scored"] - st0["candidates_scored"] == want["scored_total"]
    assert st1["sls_steps"] - st0["sls_steps"] == want["steps_total"]
    assert (want["best"] < (1 << 20)).any()       # the comparison covered complete layouts, not just the greedy build-up
    s.close()


def test_gui_weight_objective_matches_exact_minimum(eng, fixtures):
    """§8f rank 2: the GUI minimises PlatformLayout::total_weight (platform_layout.rs:174-183) under a PB bound.  The GPU
    search with the same weights reaches the minimum the oracle loop proves, with valid layouts whose total_weight is
    what the engine reports."""
    rng = np.random.default_rng(12)
    cases = [("ex1", fixtures["ex1"], O.PLATFORMS_DEFAULT, GUI_WEIGHTS), ("ex3", fixtures["ex3"], O.PLATFORMS_DEFAULT, GUI_WEIGHTS)]
    for i in range(4):
        g = (rng.random((int(rng.integers(4, 9)), int(rng.integers(4, 9)))) < 0.8).astype(np.uint8)
        defs = [(1, 1), (1, 3), (3, 3)] if i % 2 else [(1, 1), (1, 2), (2, 2)]
        w = {d: int(rng.integers(1, 6)) for d in defs}
        cases.append((f"rand{i}", g, defs, w))
    for name, grid, defs, weights in cases:
        want = oracle_min_weight(grid, defs, weights)
        wdefs = {T.PlatformDef(*d): v for d, v in weights.items()}
        res, layout, weight = eng.solve_min_weight(T.WorldGrid(grid), [T.PlatformDef(*d) for d in defs], wdefs, weight_limit=want, seed=3, max_steps=60000)
        assert res == T.SAT and weight == want, (name, weight, want)
        plats = [tup(p) for p in layout.platforms().values()]
        assert O.validate(grid, plats).is_valid
        assert O.total_weight(plats, weights) == weight == layout.total_weight(wdefs)
        if want > 0:
            res, layout, weight = eng.solve_min_weight(T.WorldGrid(grid), [T.PlatformDef(*d) for d in defs], wdefs, weight_limit=want - 1, seed=3, max_steps=3000)
            assert res == T.INTERRUPTED, name


def test_multi_platform_solver_loop_like_the_repl(eng, fixtures):
    """`load test/ex1.toml; solve` (configs[0]): default-8 set, unbounded first solve, tighten until the prover says UNSAT."""
    import ctypes as C
    from oracle.oracle import _p

    def exact(cnf):
        a = np.full(cnf.n_vars + 1, 2, np.uint8)
        lits, offs = np.ascontiguousarray(cnf.lits, np.int32), np.ascontiguousarray(cnf.offsets, np.uint32)
        r = O.lib().tsso_solve_csr(_p(lits), _p(offs, C.c_uint32), cnf.n_clauses, cnf.n_vars, _p(a, C.c_uint8), C.c_long(-1))
        return {10: T.SAT, 20: T.UNSAT}.get(r, T.INTERRUPTED), a

    g = T.WorldGrid(fixtures["ex1"])
    enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, g)
    out = T.solver_loop(T.Project(T.World(g)), enc, T.PlatformLimits(), eng, exact_solver=exact, seed=2, budget_ms=0)
    assert out["proved_optimal"] and out["best"].platform_count() == 1
    assert out["steps"][-1] == dict(bound=0, result=T.UNSAT, source="lower bound")      # optimum 1 = the packing lower bound: no proof needed
    assert all(s["source"] == "gpu" and s["valid"] for s in out["steps"][:-1])


@pytest.mark.parametrize("w,h", [(48, 40), (64, 64), (256, 256)])
def test_sls_large_grids_window_decomposition(eng, w, h):
    """C4 shape: grids larger than 32x32 are searched by window decomposition around the per-warp kernel.  The global
    layout is complete after EVERY phase (oracle validate), counts never increase, the run is deterministic, and on
    a grid that is a disjoint union of small terrains the count reaches the sum of the proven optima."""
    grid = synth_terrain(w, h, seed=1)
    g = T.WorldGrid(grid)
    counts = []
    s = eng.search(g, seed=3)
    for phase in range(6):
        s.run(1500, 0)
        counts.append(s.best_count())
        lay = s.best_layout()                               # re-validated by kernel (a) inside the engine
        if phase in (0, 5):
            sites = np.zeros((1, h, w), np.uint8)
            for p in lay.platforms().values():
                sites[0, p.y, p.x] = 1
            unc, cnt, _ = O.validate_sites_batch(grid, sites)
            assert unc[0] == 0 and cnt[0] == counts[-1]
    s.close()
    assert all(b <= a for a, b in zip(counts, counts[1:])) and counts[-1] < counts[0]
    assert counts[-1] >= -(-int(grid.sum()) // 25)
    assert counts[-1] < 0.2 * grid.sum()                    # far below "a support under every tile"
    s2 = eng.search(g, seed=3)
    for _ in range(6):
        s2.run(1500, 0)
    assert s2.best_count() == counts[-1]
    s2.close()


@pytest.mark.parametrize("w,h,seeds", [(48, 40, 8), (64, 64, 4), (70, 33, 8), (33, 90, 4)])
def test_window_decomposition_bit_exact_vs_model(eng, w, h, seeds):
    """csrc/lns.cu against its scalar replay (oracle.lns_model: frozen supports, their geodesic cover, window extraction, the
    WINDOW mode of the step rule — need mask, core-only additions — per-window winner, core write-back): the GLOBAL layout is
    the same set of supports after every phase, all four window offsets included."""
    grid = synth_terrain(w, h, seed=2, t=1)
    want = O.lns_model(grid, seeds, 5, 1200, seed=3)
    s = eng.search(T.WorldGrid(grid), seed=3, n_chains=seeds)
    for phase, (S, count) in enumerate(want):
        s.run(1200, 0)
        assert s.best_count() == count, phase
        lay = s.best_layout()
        got = np.zeros((h, w), np.uint8)
        for p in lay.platforms().values():
            got[p.y, p.x] = 1
        assert np.array_equal(got, S), phase
    s.close()


def test_sls_large_grid_reaches_sum_of_component_optima(eng, fixtures):
    """Four copies of ex3 (optimum 4 each, proven) separated by empty space on a 64x40 grid: optimum 16."""
    g = np.zeros((40, 64), np.uint8)
    e3 = fixtures["ex3"]
    for (ox, oy) in [(2, 1), (40, 3), (5, 25), (44, 28)]:
        g[oy:oy + e3.shape[0], ox:ox + e3.shape[1]] = e3
    res, lay = eng.solve_upper_bound(T.WorldGrid(g), card_limit=16, seed=1, max_steps=60000)
    assert res == T.SAT and lay.platform_count() == 16
    assert O.validate(g, [tup(p) for p in lay.platforms().values()]).is_valid
    res, lay = eng.solve_upper_bound(T.WorldGrid(g), card_limit=15, seed=1, max_steps=8000)
    assert res == T.INTERRUPTED


def test_large_grid_with_larger_platforms_merges_supports(eng):
    """Grids larger than 32x32 are searched with 1x1 supports; with a platform set that holds larger platforms the engine
    merges supports that fit under one footprint into that platform.  The result passes the reference's validate()
    (complete, footprints disjoint and in bounds), only uses platforms of the set, and needs fewer platforms than the
    1x1 layout of the same search."""
    grid = synth_terrain(96, 72, seed=4, t=1, density_q24=int(0.85 * (1 << 24)))
    g = T.WorldGrid(grid)
    counts = {}
    for name, defs in (("1x1", T.PLATFORMS_DEFAULT[:1]), ("default-8", T.PLATFORMS_DEFAULT)):
        s = eng.search(g, defs, seed=5)
        for _ in range(4):
            s.run(1500, 0)
        lay = s.best_layout()                                   # re-validated by kernel (a) (platform evaluator) inside the engine
        s.close()
        plats = list(lay.platforms().values())
        assert O.validate(grid, [tup(p) for p in plats]).is_valid
        assert all(p.definition in defs for p in plats)
        counts[name] = len(plats)
    assert counts["default-8"] < 0.8 * counts["1x1"]
    res, lay = eng.solve_upper_bound(g, T.PLATFORMS_DEFAULT, seed=5, max_steps=3000)
    assert res == T.SAT and O.validate(grid, [tup(p) for p in lay.platforms().values()]).is_valid and lay.platform_count() < 0.8 * counts["1x1"]


def test_solve_batch_terrains(eng):
    """C5 shape (scaled down): per-terrain counts are complete layouts, never below the trivial lower bound, and
    agree with the oracle's proven optimum where that is cheap to prove."""
    n = 96
    grids = np.stack([synth_terrain(32, 32, seed=1, t=t) for t in range(n)])
    counts, layouts = eng.solve_batch(grids, seed=1, steps=3000, want_layouts=True)
    assert (counts > 0).all()
    sites = ((layouts[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8)
    for t in range(0, n, 7):
        unc, cnt, _ = O.validate_sites_batch(grids[t], sites[t][None])
        assert unc[0] == 0 and cnt[0] == counts[t]
        assert counts[t] >= -(-int(grids[t].sum()) // 25)
    # the batch is the step rule of the spec, terrain by terrain: chains 4t .. 4t+3 of the seed, the bound shared every 1024 steps —
    # the oracle's flat-array CPU port (the bench's CPU arm for configs[4]) run that way reports the same count for every terrain
    for t in range(0, n, 5):
        r = O.sls_flat(grids[t], 4, [(1024, 1 << 20, 0), (1024, 1 << 20, 0), (952, 1 << 20, 0)], seed=1, chain_offset=4 * t, want_layouts=False)
        assert int(r["best"].min()) == counts[t], t
    small = np.stack([synth_terrain(8, 8, seed=3, t=t) for t in range(12)])
    c2 = eng.solve_batch(small, seed=1, steps=2000)
    for t in range(12):
        r = O.solver_loop(small[t], O.PLATFORMS_1X1)
        assert r["proved_optimal"] and c2[t] == len(r["best"]), t


def test_c5_full_size_batch_properties(eng):
    """BASELINE.json configs[4] at full size: 100 000 synthetic 32x32 terrains through tss_solve_batch.  Too many for
    the oracle, so: every reported layout is re-evaluated by kernel (a) in per-terrain mode (complete, count matches),
    counts respect the trivial lower bound ceil(tiles/25), the run is deterministic, and a sample is validated by the
    oracle."""
    import torch
    n = 100_000
    lib = T.load()
    grids = np.zeros((n, 32, 32), np.uint8)
    import ctypes as C
    for t in range(n):
        lib.tss_world_synthetic(32, 32, 1, t, int(0.7 * (1 << 24)), grids[t].ctypes.data_as(C.POINTER(C.c_uint8)))
    counts, layouts = eng.solve_batch(grids, seed=1, steps=1500, want_layouts=True)
    assert counts.shape == (n,) and (counts > 0).all()
    tiles = grids.reshape(n, -1).sum(1).astype(np.int64)
    assert (counts >= (tiles + 24) // 25).all() and (counts <= tiles).all()
    # per-terrain re-evaluation on the device (kernel a, per_layout_terrain): terrain rows and layout rows are both u32[32]
    terr_rows = pack_rows(grids).reshape(n, 32)
    g_dev = torch.from_numpy(terr_rows.view(np.int32)).cuda()
    l_dev = torch.from_numpy(layouts.view(np.int32)).cuda()
    out = torch.empty((n, 2), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    eng.eval_compact_dev(g_dev.data_ptr(), 32, 32, l_dev.data_ptr(), n, out.data_ptr(), per_layout_terrain=True)
    torch.cuda.synchronize()   # device-wide: also waits for the engine's own stream
    res = out.cpu().numpy()
    assert (res[:, 0] == 0).all() and np.array_equal(res[:, 1], counts)
    sites = ((layouts[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).astype(np.uint8)
    for t in (0, 31337, 99_999):
        unc, cnt, _ = O.validate_sites_batch(grids[t], sites[t][None])
        assert unc[0] == 0 and cnt[0] == counts[t]
    again = eng.solve_batch(grids[:4096], seed=1, steps=1500)
    assert np.array_equal(again, counts[:4096])


def test_solver_loop_gpu_then_exact_proof(eng, fixtures):
    """crates/repl/src/main.rs:280-366 with the GPU as the SAT side and the oracle's CDCL as the Glucose stand-in:
    the loop ends with UNSAT one below the GPU's count, i.e. the GPU reached the proven optimum."""
    def exact(cnf):
        import ctypes as C
        a = np.full(cnf.n_vars + 1, 2, np.uint8)
        clauses = [list(map(int, c)) for c in cnf.clauses()]
        h = O.lib()
        # route the product's CNF through the oracle's solver entry (DIMACS arrays in, model out)
        from oracle.oracle import _p
        lits = np.ascontiguousarray(cnf.lits, np.int32)
        offs = np.ascontiguousarray(cnf.offsets, np.uint32)
        h.tsso_solve_csr.restype = C.c_int
        r = h.tsso_solve_csr(_p(lits), _p(offs, C.c_uint32), cnf.n_clauses, cnf.n_vars, _p(a, C.c_uint8), C.c_long(-1))
        return {10: T.SAT, 20: T.UNSAT}.get(r, T.INTERRUPTED), a

    for name, optimum in KNOWN_OPTIMA[:2]:
        g = T.WorldGrid(fixtures[name])
        proj = T.Project(T.World(g))
        enc = T.Encoding.encode(T.PLATFORMS_DEFAULT[:1], g)
        out = T.solver_loop(proj, enc, T.PlatformLimits(), eng, exact_solver=exact, seed=1, budget_ms=0, use_lower_bound=False)
        assert out["proved_optimal"] and out["best"].platform_count() == optimum
        assert all(s["valid"] for s in out["steps"] if s["result"] == T.SAT)
        assert out["steps"][-1]["result"] == T.UNSAT and out["steps"][-1]["source"] == "exact"
        assert [s["source"] for s in out["steps"][:-1]] == ["gpu"] * (len(out["steps"]) - 1)


# =============================================================================== packing lower bound (tss_lower_bound)
def _key_dims(defs):
    out = []
    for d in defs:      # dims keys: defs order, unflipped then flipped (src/encoder.rs:121-130)
        for dims in ((d.width, d.height), (d.height, d.width)):
            if dims not in out:
                out.append(dims)
    return out


def _check_packing(g, defs, tiles):
    """The bound's witness against the reference's own rule: every in-bounds placement of every dims key, validated ALONE by
    the oracle's validate() (platform_layout.rs:85-149), supports at most one packed tile — so a layout needs >= len(tiles)."""
    h, w = g.shape
    packed = np.zeros_like(g)
    for x, y in tiles:
        assert g[y, x] == 1                                  # ceiling tiles only
        packed[y, x] = 1
    assert packed.sum() == len(tiles)
    for kw, kh in _key_dims(defs):
        for y in range(h - kh + 1):
            for x in range(w - kw + 1):
                plat = (x, y, min(kw, kh), max(kw, kh), int(kw > kh))
                v = O.validate(g, [plat])
                assert not v.out_of_bounds
                supported = g & (1 - v.unsupported)
                assert int((supported & packed).sum()) <= 1, (plat, tiles)


@pytest.mark.parametrize("name", ["ex1", "ex3", "ex2", "rect8", "rand20x14"])
@pytest.mark.parametrize("pset", ["1x1", "default8", "1x1+3x3"])
def test_lower_bound_packing_is_sound(eng, fixtures, name, pset):
    g = {"rect8": np.ones((8, 8), np.uint8), "rand20x14": synth_terrain(20, 14, seed=3, t=1)}.get(name)
    if g is None:
        g = fixtures[name]
    defs = {"1x1": T.PLATFORMS_DEFAULT[:1], "default8": T.PLATFORMS_DEFAULT, "1x1+3x3": (T.PlatformDef(1, 1), T.PlatformDef(3, 3))}[pset]
    tiles = eng.lower_bound(T.WorldGrid(g), defs, seed=1)
    assert len(tiles) >= 1
    _check_packing(g, defs, tiles)
    key = f"{name}/{pset}"
    proofs = golden("proofs")
    if key in proofs:
        assert len(tiles) <= proofs[key]["optimum"]          # a lower bound never exceeds the proven optimum
    # the bound is monotone in the platform set: more platform types can only lower it
    if pset != "1x1":
        assert len(tiles) <= len(eng.lower_bound(T.WorldGrid(g), T.PLATFORMS_DEFAULT[:1], seed=1))


def test_lower_bound_edge_cases(eng):
    assert eng.lower_bound(T.WorldGrid(np.zeros((4, 5), np.uint8))) == []                         # no ceiling: nothing to support
    assert eng.lower_bound(T.WorldGrid(np.ones((1, 1), np.uint8))) == [(0, 0)]
    two = np.zeros((1, 32), np.uint8)
    two[0, 0] = two[0, 31] = 1                                                                    # two islands: one support each
    assert sorted(eng.lower_bound(T.WorldGrid(two))) == [(0, 0), (31, 0)]
    line = np.ones((1, 32), np.uint8)                                                             # a corridor: tiles 7 apart, ceil(32/7) = 5
    tiles = eng.lower_bound(T.WorldGrid(line))
    assert len(tiles) == 5 and all(b[0] - a[0] >= 7 for a, b in zip(sorted(tiles), sorted(tiles)[1:]))
    tall = eng.lower_bound(T.WorldGrid(np.ones((33, 8), np.uint8)))                               # beyond 32 rows: the whole-board kernel
    assert len(tall) >= 4 and all(abs(a[0] - b[0]) + abs(a[1] - b[1]) > 6 for i, a in enumerate(tall) for b in tall[:i])
    with pytest.raises(T.TssError):
        eng.lower_bound(T.WorldGrid(np.ones((600, 600), np.uint8)))                               # boards beyond 256x256 do not fit shared memory
    full = np.ones((32, 32), np.uint8)
    tiles = eng.lower_bound(T.WorldGrid(full))
    assert len(tiles) >= 32 * 32 // 85 + 1 and len(tiles) <= 41                                   # radius-6 balls hold <= 85 tiles; optimum >= 1024/25


def _check_lp_certificate(g, defs, r):
    """The fractional bound's certificate against the reference's own rule, in exact integer arithmetic: the weights are
    non-negative and sit on ceiling tiles, NO in-bounds placement — validated alone by the oracle's validate()
    (platform_layout.rs:85-149) — supports more than max_load of them, and the bound is ceil(total / max_load)."""
    h, w = g.shape
    wts = r["weights"].astype(np.int64)
    assert (wts >= 0).all() and (wts[g == 0] == 0).all() and int(wts.sum()) == r["total"]
    worst = 0
    for kw, kh in _key_dims(defs):
        for y in range(h - kh + 1):
            for x in range(w - kw + 1):
                v = O.validate(g, [(x, y, min(kw, kh), max(kw, kh), int(kw > kh))])
                supported = (g & (1 - v.unsupported)).astype(bool)
                worst = max(worst, int(wts[supported].sum()))
    assert worst == r["max_load"] > 0
    assert r["bound"] == -(-r["total"] // r["max_load"])


def _platform_cost(kw, kh, weights):
    """what PlatformLayout::total_weight charges one platform: the weights of every def that fits inside its def (platform_layout.rs:174-183)"""
    cw, ch = min(kw, kh), max(kw, kh)
    return sum(v for (dw, dh), v in weights.items() if min(dw, dh) <= cw and max(dw, dh) <= ch)


def test_fractional_lower_bound_on_the_gui_weight_objective(eng, fixtures):
    """crates/gui/src/app.rs:235-245 minimises total_weight.  The weighted certificate, re-derived placement by placement with the
    oracle's validate(): bound = min over placements of ceil(total * cost / load); it never exceeds the minimum weight the oracle's
    GUI loop proves, and the GPU-seeded GUI loop (api.weight_loop) reaches that minimum — without the exact solver where the
    bound meets it."""
    rng = np.random.default_rng(12)
    cases = [("ex1", fixtures["ex1"], O.PLATFORMS_DEFAULT, GUI_WEIGHTS), ("ex3", fixtures["ex3"], O.PLATFORMS_DEFAULT, GUI_WEIGHTS)]
    for i in range(3):
        g = (rng.random((int(rng.integers(4, 9)), int(rng.integers(4, 9)))) < 0.8).astype(np.uint8)
        defs = [(1, 1), (1, 3), (3, 3)] if i % 2 else [(1, 1), (1, 2), (2, 2)]
        cases.append((f"rand{i}", g, defs, {d: int(rng.integers(1, 6)) for d in defs}))

    def exact(cnf):
        import ctypes as C
        a = np.full(cnf.n_vars + 1, 2, np.uint8)
        lits, offs = np.ascontiguousarray(cnf.lits, np.int32), np.ascontiguousarray(cnf.offsets, np.uint32)
        r = O.lib().tsso_solve_csr(O._p(lits), O._p(offs, C.c_uint32), cnf.n_clauses, cnf.n_vars, O._p(a, C.c_uint8), C.c_long(-1))
        return {10: T.SAT, 20: T.UNSAT}.get(r, T.INTERRUPTED), a

    closed = 0
    for name, g, defs, weights in cases:
        h, w = g.shape
        tdefs = [T.PlatformDef(*d) for d in defs]
        wdefs = {T.PlatformDef(*d): v for d, v in weights.items()}
        r = eng.lower_bound_lp(T.WorldGrid(g), tdefs, weights=wdefs)
        wts = r["weights"].astype(np.int64)
        assert (wts >= 0).all() and (wts[g == 0] == 0).all() and int(wts.sum()) == r["total"]
        best = None
        for kw, kh in _key_dims(tdefs):
            cost = _platform_cost(kw, kh, weights)
            for y in range(h - kh + 1):
                for x in range(w - kw + 1):
                    v = O.validate(g, [(x, y, min(kw, kh), max(kw, kh), int(kw > kh))])
                    load = int(wts[(g & (1 - v.unsupported)).astype(bool)].sum())
                    if load > 0:
                        q = -(-(r["total"] * cost) // load)
                        best = q if best is None else min(best, q)
        assert r["bound"] == best, name
        want = oracle_min_weight(g, defs, weights)
        assert r["bound"] <= want, (name, r["bound"], want)
        grid = T.WorldGrid(g)
        out = T.weight_loop(T.Project(T.World(grid)), T.Encoding.encode(tdefs, grid), wdefs, eng, exact_solver=exact, seed=2)
        assert out["proved_optimal"] and out["best_weight"] == want, (name, out["best_weight"], want, out["steps"])
        plats = [tup(p) for p in out["best"].platforms().values()]
        assert O.validate(g, plats).is_valid and O.total_weight(plats, weights) == want
        closed += out["steps"][-1]["source"] == "lower bound"
    print("GUI loops closed by the certified bound alone:", closed, "of", len(cases))


@pytest.mark.parametrize("name", ["ex1", "ex3", "ex2", "readme", "rect16", "rand20x14", "rect24"])
@pytest.mark.parametrize("pset", ["1x1", "default8"])
def test_fractional_lower_bound_certificate(eng, fixtures, readme, name, pset):
    g = {"rect16": np.ones((16, 16), np.uint8), "rect24": np.ones((24, 24), np.uint8), "rand20x14": synth_terrain(20, 14, seed=3, t=1), "readme": readme[0]}.get(name)
    if g is None:
        g = fixtures[name]
    defs = T.PLATFORMS_DEFAULT[:1] if pset == "1x1" else T.PLATFORMS_DEFAULT
    r = eng.lower_bound_lp(T.WorldGrid(g), defs)
    assert r["optimal"] and r["pivots"] > 0
    _check_lp_certificate(g, defs, r)
    assert r["bound"] >= len(eng.lower_bound(T.WorldGrid(g), defs, seed=1))       # the LP relaxes the integral packing
    proofs = golden("proofs")
    key = f"{name}/{pset}"
    if key in proofs:
        assert r["bound"] <= proofs[key]["optimum"]
    # SURVEY.md configs[2] and test/ex2.toml with 1x1 supports: the fractional bound IS the optimum (LP value 13.13 / 13.2 -> 14),
    # the integral packing stops at 12 / 13; rect 16x16: 14 of 15
    want = {"readme/1x1": 14, "ex2/1x1": 14, "rect16/1x1": 14, "ex1/1x1": 3, "ex3/1x1": 4, "ex2/default8": 4}.get(key)
    if want is not None:
        assert r["bound"] == want
    # target: stop as soon as the bound reaches it — fewer pivots, the same answer to "does the bound reach r?", still certified;
    # a target above the LP optimum runs to optimality
    early = eng.lower_bound_lp(T.WorldGrid(g), defs, target=r["bound"])
    assert early["bound"] == r["bound"] and early["pivots"] <= r["pivots"]
    _check_lp_certificate(g, defs, early)
    if name in ("ex2", "readme", "rect16") and pset == "1x1":
        assert early["pivots"] < r["pivots"] and not early["optimal"]
    beyond = eng.lower_bound_lp(T.WorldGrid(g), defs, target=r["bound"] + 1)
    assert beyond["optimal"] and beyond["bound"] == r["bound"]
    capped = eng.lower_bound_lp(T.WorldGrid(g), defs, max_pivots=5)                # an iteration cap only weakens the bound, it stays certified
    assert not capped["optimal"] or capped["pivots"] <= 5
    _check_lp_certificate(g, defs, capped)
    assert capped["bound"] <= r["bound"]


def test_solver_loop_proves_readme_and_ex2_without_the_exact_solver(eng, fixtures, readme):
    """BASELINE.json configs[2] (README terrain, 1x1 supports, "proven-optimal count match") and test/ex2.toml: SLS reaches 14, the
    certified fractional bound is 14 — the loop ends proven optimal with no exact-solver call (the reference's Glucose, and
    the CDCL stand-in here, spend their time on exactly that last UNSAT call: 10 s and more, tests/golden/proofs.json)."""
    def exact(cnf):
        raise AssertionError("the exact solver must not be needed")

    for name, g in (("readme", readme[0]), ("ex2", fixtures["ex2"])):
        grid = T.WorldGrid(g)
        enc = T.Encoding.encode(T.PLATFORMS_DEFAULT[:1], grid)
        out = T.solver_loop(T.Project(T.World(grid)), enc, T.PlatformLimits(), eng, exact_solver=exact, seed=6)
        assert out["proved_optimal"] and out["best"].platform_count() == golden("proofs")[f"{name}/1x1"]["optimum"] == out["lower_bound"] == 14
        assert out["steps"][-1]["source"] == "lower bound"
        plats = [tup(p) for p in out["best"].platforms().values()]
        assert O.validate(g, plats).is_valid


def _geodesic_ball(g, x, y, radius):
    cur = np.zeros_like(g, dtype=bool)
    cur[y, x] = True
    c = g.astype(bool)
    for _ in range(radius):
        n = cur.copy()
        n[1:] |= cur[:-1]; n[:-1] |= cur[1:]; n[:, 1:] |= cur[:, :-1]; n[:, :-1] |= cur[:, 1:]
        cur = n & c
    return cur


@pytest.mark.parametrize("w,h", [(96, 80), (33, 40), (256, 256)])
def test_lower_bound_on_large_grids(eng, w, h):
    """Grids beyond 32x32 (C4's shape), 1x1 supports: the whole-board packing.  Independent check in numpy: the packed tiles are
    ceiling tiles pairwise more than 6 steps apart through the ceiling (= no site within 3 of two of them: validate()'s three
    dilations, platform_layout.rs:127-141), and the bound is useful (well above tiles / 25, below the SLS count)."""
    g = synth_terrain(w, h, seed=1, t=0 if (w, h) == (256, 256) else 3)
    tiles = eng.lower_bound(T.WorldGrid(g), seed=1)
    packed = np.zeros_like(g, dtype=bool)
    for x, y in tiles:
        assert g[y, x] == 1
        packed[y, x] = True
    assert packed.sum() == len(tiles)
    sample = tiles if len(tiles) <= 400 else [tiles[i] for i in np.random.default_rng(0).choice(len(tiles), 400, replace=False)]
    for x, y in sample:
        assert (_geodesic_ball(g, x, y, 6) & packed).sum() == 1, (x, y)
    assert len(tiles) > 1.5 * g.sum() / 25                     # far better than the trivial ceil(tiles / 25)
    if (w, h) == (96, 80):
        s = eng.search(T.WorldGrid(g), seed=2)
        for _ in range(4):
            s.run(2000, 0)
        assert len(tiles) <= s.best_count()
        s.close()
    with pytest.raises(T.TssError):
        eng.lower_bound(T.WorldGrid(g), T.PLATFORMS_DEFAULT)    # larger platform sets: grids up to 32x32 only


def test_solver_loop_ends_on_the_lower_bound_without_the_exact_solver(eng, fixtures):
    """BASELINE.json configs[0]: the REPL's own run (default-8 set) on test/ex1.toml and ex3.toml — optimum 1, and any ceiling
    tile is a packing of size 1: the loop is finished by the GPU alone, the exact solver is never called."""
    calls = []

    def exact(cnf):
        calls.append(cnf.n_vars)
        raise AssertionError("the exact solver must not be needed")

    for name in ("ex1", "ex3"):
        g = T.WorldGrid(fixtures[name])
        enc = T.Encoding.encode(T.PLATFORMS_DEFAULT, g)
        out = T.solver_loop(T.Project(T.World(g)), enc, T.PlatformLimits(), eng, exact_solver=exact, seed=4)
        assert out["proved_optimal"] and out["best"].platform_count() == golden("proofs")[f"{name}/default8"]["optimum"] == out["lower_bound"] == 1
        assert out["steps"][-1]["source"] == "lower bound" and not calls
        assert all(s["valid"] for s in out["steps"] if s["result"] == T.SAT)


# =============================================================================== the C++ driver over the C ABI (tools/tss_repl.cpp)
def _run_repl(tmp_path, grid, *args):
    import subprocess
    import sys
    proj = tmp_path / "project.toml"
    proj.write_text(T.WorldGrid(grid).to_toml())
    exe = os.path.join(os.path.dirname(T.__file__), "tss_repl")
    exact = f"{sys.executable} {os.path.join(os.path.dirname(__file__), 'exact_dimacs.py')}"
    out = subprocess.run([exe, str(proj), "--exact", exact, *args], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    summary = [ln for ln in out.stdout.splitlines() if ln.startswith("# best=")][-1]
    import re
    fields = dict(kv.split("=", 1) for kv in re.sub(r'verdict="[^"]*" ', "", summary[2:]).split(" ") if "=" in kv)
    fields["verdict"] = re.search(r'verdict="([^"]*)"', summary).group(1)
    counts = [int(ln.split("(")[1].split()[0]) for ln in out.stdout.splitlines() if ln.startswith("Solution found")]
    return out.stdout, fields, counts


@pytest.mark.parametrize("name,pset,key", [("ex1", "default", "ex1/default8"), ("ex3", "default", "ex3/default8"), ("ex2", "default", "ex2/default8"),
                                           ("ex1", "1x1", "ex1/1x1"), ("ex3", "1x1", "ex3/1x1")])
def test_cpp_repl_driver_reaches_the_proven_optimum(eng, fixtures, tmp_path, name, pset, key):
    """BASELINE.json configs[0]: `load test/exN.toml; solve` through tools/tss_repl.cpp — the REPL's loop (main.rs:280-366) in C++
    over the C ABI, performing the Rust shim's call sequence (upload the clauses, find the instance from them, SAT-like GPU
    solve, witness verified against those clauses), the oracle CDCL standing in for Glucose as `--exact`.  It must end with
    the proven optimum, strictly decreasing counts (bound = found - 1), and the REPL's closing lines."""
    optimum = golden("proofs")[key]["optimum"]
    text, f, counts = _run_repl(tmp_path, fixtures[name], "--platforms", pset, "--seed", "3")
    assert int(f["best"]) == optimum and counts[-1] == optimum
    assert all(b < a for a, b in zip(counts, counts[1:]))
    assert "No solution found for the current constraints" in text and text.rstrip().splitlines()[-2] == "Done"
    assert f["verdict"].startswith("optimal") and "FAILED" not in text
    # tss_solve_instance answers UNSAT below the certified lower bounds, which are tight on all five: the exact solver is never started
    assert int(f["exact_solves"]) == 0 and int(f["lower_bound"]) == optimum and f["verdict"] == "optimal (lower bound)"
    # ... and with the bound-based answers switched off the same loop ends on the exact solver's UNSAT
    text, f, counts = _run_repl(tmp_path, fixtures[name], "--platforms", pset, "--seed", "3", "--no-lower-bound")
    assert int(f["best"]) == optimum and int(f["exact_solves"]) >= 1 and f["verdict"] == "optimal (exact solver)"


@pytest.mark.parametrize("name", ["ex1", "ex3"])
def test_cpp_driver_runs_the_gui_weight_loop(eng, fixtures, tmp_path, name):
    """crates/gui/src/app.rs:212-249 through tools/tss_repl.cpp --gui: default-8 set with the GUI's default weights, weight_limit =
    total_weight - 1 after every solution, until Unsat — over the C ABI with the shim's call sequence (the instance registry hands
    the weights back, tss_solve_instance steers by the weight limit, the witness satisfies the PB constraint's clauses, and the
    weighted fractional bound answers UNSAT where it meets the weight).  The final weight is the minimum the oracle's GUI loop proves."""
    want = oracle_min_weight(fixtures[name], O.PLATFORMS_DEFAULT, GUI_WEIGHTS)
    text, f, counts = _run_repl(tmp_path, fixtures[name], "--gui", "--seed", "3")
    weights = [int(ln.split()[-1]) for ln in text.splitlines() if ln.startswith("Got a solution with weight")]
    assert int(f["weight"]) == want == weights[-1] and all(b < a for a, b in zip(weights, weights[1:]))
    assert f["verdict"].startswith("optimal") and "FAILED" not in text and int(f["gpu_solves"]) >= 2
    if f["verdict"] == "optimal (lower bound)":
        assert int(f["exact_solves"]) == 0 and int(f["lower_bound"]) == want
    # ... and with the bound-based answers switched off the exact solver proves the same minimum
    text, f, counts = _run_repl(tmp_path, fixtures[name], "--gui", "--seed", "3", "--no-lower-bound")
    assert int(f["weight"]) == want and f["verdict"] == "optimal (exact solver)" and int(f["exact_solves"]) >= 1


def test_cpp_repl_driver_limits_and_errors(eng, fixtures, tmp_path):
    # `solve -l 1:2` on ex1 with 1x1 supports: 3 are needed (proofs.json) -> UNSAT straight from the exact solver
    text, f, counts = _run_repl(tmp_path, fixtures["ex1"], "--platforms", "1x1", "-l", "1:2", "--no-lower-bound")
    assert counts == [] and f["verdict"] == "unsatisfiable" and int(f["exact_solves"]) == 1
    text, f, counts = _run_repl(tmp_path, fixtures["ex1"], "--platforms", "1x1", "-l", "1:2")   # ... or from the certified bound: no exact solver
    assert counts == [] and f["verdict"] == "unsatisfiable" and int(f["exact_solves"]) == 0 and "No solution found" in text
    # a limit on another platform type is left to the exact solver (the search cannot steer by it), and still honoured
    text, f, counts = _run_repl(tmp_path, fixtures["ex1"], "-l", "5:0,3:0")
    assert int(f["best"]) >= 2 and int(f["gpu_solves"]) >= 1 and int(f["exact_solves"]) >= 1
    import subprocess
    exe = os.path.join(os.path.dirname(T.__file__), "tss_repl")
    bad = tmp_path / "bad.toml"
    bad.write_text('[world]\ngrid = ["XZ"]\n')
    r = subprocess.run([exe, str(bad)], capture_output=True, text=True)
    assert r.returncode == 1 and "Error parsing file" in r.stderr                   # src/world.rs:49-79: any other character is an error


def test_interrupt_returns_unknown(eng):
    g = T.WorldGrid(np.ones((16, 16)))
    eng.interrupt()
    res, layout = eng.solve_upper_bound(g, card_limit=14, seed=1, budget_ms=2000)
    eng.clear_interrupt()
    assert res == T.INTERRUPTED and eng.stats()["interrupted"] == 1


def test_errors_and_edge_cases(eng):
    with pytest.raises(T.TssError) as e:
        eng.search(T.WorldGrid(np.ones((4, 4))), defs=[T.PlatformDef(3, 3)])
    assert e.value.code == -1                                                    # no 1x1 in the platform set
    res, layout = eng.solve_upper_bound(T.WorldGrid(np.zeros((5, 5))), seed=1, max_steps=100)
    assert res == T.SAT and layout.platform_count() == 0                         # no ceiling: the empty layout
    res, layout = eng.solve_upper_bound(T.WorldGrid(rows_to_grid(["X X X X"])), seed=1, max_steps=1000)
    assert res == T.SAT and layout.platform_count() == 4                         # isolated tiles need one support each
    unc, cnt = eng.eval_sites(T.WorldGrid(np.ones((3, 3))), np.zeros((0, 3, 3), np.uint8))
    assert len(unc) == 0


def test_c_abi_from_plain_c(tmp_path):
    """The boundary from a C host: tests/c_abi_smoke.c (gcc, no Python in the loop) loads a project, solves with the
    REPL's platform set, validates, checks the witness against the encoder's CNF, exercises the error and interrupt paths."""
    import subprocess
    from test_host import build_c_abi_smoke
    out = subprocess.run([build_c_abi_smoke(tmp_path)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert "c_abi_smoke ok" in out.stdout


def test_measured_peaks_sane(eng):
    p = eng.measure_peaks()
    sm = eng.device_info()["sm_count"]
    assert 500 < p["sm_mhz"] < 2500
    # LOP3: at most 64 lanes/clk/SM (alu pipe, 16 lanes per SMSP) .. allow the 128-lane case too
    assert 0.2 * 64 * sm * p["sm_mhz"] / 1e3 < p["lop3_gops"] < 1.1 * 128 * sm * p["sm_mhz"] / 1e3
    assert p["popc_gops"] > 0 and p["shfl_gops"] > 0 and p["smem_gbs"] > 1000


def test_error_paths_return_codes_not_crashes(eng):
    """Error behaviour at the boundary (SURVEY.md §8b): status codes + tss_last_error, never an abort."""
    import ctypes as C
    lib = T.load()
    g = np.ones((4, 4), np.uint8)
    gp = g.ctypes.data_as(C.POINTER(C.c_uint8))
    n = C.c_int32()
    assert lib.tss_solve_upper_bound(eng._h, None, 4, 4, None, 0, -1, 0, 0, 10, None, 0, C.byref(n)) == -1       # null grid
    assert lib.tss_solve_upper_bound(eng._h, gp, 0, 4, None, 0, -1, 0, 0, 10, None, 0, C.byref(n)) == -1          # zero-sized grid
    assert b"bad arguments" in lib.tss_last_error(eng._h)
    big = np.ones((700, 700), np.uint8)
    with pytest.raises(T.TssError) as e:
        eng.search(T.WorldGrid(big))
    assert e.value.code == -4                                                                                    # TSS_E_UNSUPPORTED
    lits = np.array([1, -9], np.int32)
    offs = np.array([0, 2], np.uint32)
    h = C.c_void_p()
    assert lib.tss_cnf_upload(eng._h, lits.ctypes.data_as(C.POINTER(C.c_int32)), offs.ctypes.data_as(C.POINTER(C.c_uint32)), 1, 3, C.byref(h)) == -1
    assert b"out of range" in lib.tss_last_error(eng._h)
    with pytest.raises(T.TssError):
        eng.solve_min_weight(T.WorldGrid(g), T.PLATFORMS_DEFAULT[:1], {T.PlatformDef(1, 1): 5})                  # weight objective needs > 1 key
    s = eng.search(T.WorldGrid(g), seed=1, n_chains=8)
    with pytest.raises(T.TssError):
        s.best_layout()                                                                                          # nothing found yet
    with pytest.raises(T.TssError):
        s.run(0, 0)
    s.close()
    assert eng.comm_world() == 1
