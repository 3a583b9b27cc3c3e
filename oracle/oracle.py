"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/_build/libtss_oracle.so (the CPU restatement of the reference's
feasibility-and-bound path, see oracle/oracle.hpp).  Importable only from tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs; the product package
never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libtss_oracle.so")

PLATFORMS_1X1 = [(1, 1)]
PLATFORMS_DEFAULT = [(1, 1), (1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (3, 3), (5, 5)]  # src/platform.rs:23-32
FAMILIES = ["dag_impl", "dag_sibling", "t3_platform", "layer", "unit_t0", "overlap_anchor", "overlap_cross",
            "oob", "limit_link", "card", "pb"]


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".cpp", ".hpp"))]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        L = _lib
        L.tsso_encode.restype = C.c_void_p
        L.tsso_encoding_cnf.restype = C.c_void_p
        L.tsso_with_limits.restype = C.c_void_p
        L.tsso_cnf_num_lits.restype = C.c_long
        L.tsso_total_weight.restype = C.c_long
        L.tsso_assignment_total_weight.restype = C.c_long
        L.tsso_validate_sites_batch.restype = C.c_double
    return _lib


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a, t=C.c_int):
    return a.ctypes.data_as(C.POINTER(t))


def _grid(grid):
    g = np.ascontiguousarray(grid, dtype=np.uint8)
    assert g.ndim == 2
    return g


# --------------------------------------------------------------------------- math / platform
def dims_partial_cmp(a, b):
    r = lib().tsso_dims_partial_cmp(a[0], a[1], b[0], b[1])
    return None if r == 2 else r


def iter_within(w, h):
    out = np.zeros((w * h + 1, 2), np.int32)
    n = lib().tsso_iter_within(w, h, _p(out), len(out))
    return [tuple(map(int, p)) for p in out[:n]]


def iter_manhattan(c, dist):
    out = np.zeros((4 * (dist + 1) ** 2, 2), np.int32)
    n = lib().tsso_iter_manhattan(c[0], c[1], dist, _p(out), len(out))
    return [tuple(map(int, p)) for p in out[:n]]


def neighbors(p):
    out = np.zeros((4, 2), np.int32)
    lib().tsso_neighbors(p[0], p[1], _p(out))
    return [tuple(map(int, q)) for q in out]


def platform_overlaps(a, b):
    """a, b: (x, y, def_w, def_h, rotated)"""
    return bool(lib().tsso_platform_overlaps(_p(_i32(a)), _p(_i32(b))))


# --------------------------------------------------------------------------- world
class WorldParseError(ValueError):
    pass


def parse_world(text: str):
    """-> (grid uint8[h, w], ragged)"""
    out = np.zeros(1 << 22, np.uint8)
    w, h, rg = C.c_int(), C.c_int(), C.c_int()
    err = C.create_string_buffer(512)
    r = lib().tsso_parse_world(text.encode(), _p(out, C.c_uint8), len(out), C.byref(w), C.byref(h), C.byref(rg), err, 512)
    if r != 0:
        raise WorldParseError(err.value.decode() or "grid too large")
    return out[: w.value * h.value].reshape(h.value, w.value).copy(), bool(rg.value)


def world_to_toml(grid) -> str:
    g = _grid(grid)
    buf = C.create_string_buffer(g.size * 2 + 64 * g.shape[0] + 64)
    n = lib().tsso_world_to_toml(_p(g, C.c_uint8), g.shape[1], g.shape[0], buf, len(buf))
    assert n >= 0
    return buf.value.decode()


def dag_edges(defs):
    d = _i32(defs)
    out = np.zeros((256, 4), np.int32)
    n = lib().tsso_dag_platform_edges(_p(d), len(d), _p(out), len(out))
    plat = [((int(a), int(b)), (int(c), int(e))) for a, b, c, e in out[:n]]
    n = lib().tsso_dag_point_edges(_p(d), len(d), _p(out), len(out))
    pts = [((int(a), int(b)), (int(c), int(e))) for a, b, c, e in out[:n]]
    return plat, pts


# --------------------------------------------------------------------------- CNF
def propagate_csr(lits, offsets, n_vars, assignment):
    """Unit propagation (synchronous rounds, oracle/capi.cpp) on a caller-provided CSR CNF -> (assignment, conflict clause or -1, rounds)."""
    lits = np.ascontiguousarray(lits, np.int32)
    offsets = np.ascontiguousarray(offsets, np.uint32)
    a = np.ascontiguousarray(assignment, dtype=np.uint8).copy()
    conflict, rounds = C.c_int(), C.c_int()
    lib().tsso_propagate_csr(_p(lits if len(lits) else np.zeros(1, np.int32)), _p(offsets, C.c_uint32), len(offsets) - 1, n_vars, _p(a, C.c_uint8), C.byref(conflict), C.byref(rounds))
    return a, conflict.value, rounds.value


class Cnf:
    def __init__(self, handle):
        self._h = C.c_void_p(handle)
        L = lib()
        self.n_vars = L.tsso_cnf_num_vars(self._h)
        self.n_clauses = L.tsso_cnf_num_clauses(self._h)
        self.n_lits = L.tsso_cnf_num_lits(self._h)
        self.lits = np.zeros(max(self.n_lits, 1), np.int32)
        self.offsets = np.zeros(self.n_clauses + 1, np.uint32)
        self.family = np.zeros(max(self.n_clauses, 1), np.uint8)
        L.tsso_cnf_get(self._h, _p(self.lits), _p(self.offsets, C.c_uint32), _p(self.family, C.c_uint8))
        self.lits = self.lits[: self.n_lits]
        self.family = self.family[: self.n_clauses]

    def __del__(self):
        if lib is not None and self._h:
            lib().tsso_cnf_free(self._h)
            self._h = None

    def clauses(self):
        o = self.offsets
        return [tuple(int(x) for x in self.lits[o[i]: o[i + 1]]) for i in range(self.n_clauses)]

    def family_counts(self):
        return {FAMILIES[f]: int((self.family == f).sum()) for f in np.unique(self.family)}

    def solve(self, conflict_budget=-1):
        """-> (result 10/20/0, assignment uint8[n_vars+1] or None, stats dict)"""
        a = np.full(self.n_vars + 1, 2, np.uint8)
        st = (C.c_ulonglong * 5)()
        sec = C.c_double()
        r = lib().tsso_cnf_solve(self._h, _p(a, C.c_uint8), C.c_long(conflict_budget), None, st, C.byref(sec))
        stats = dict(conflicts=st[0], decisions=st[1], propagations=st[2], restarts=st[3], learnts=st[4], seconds=sec.value)
        return r, (a if r == 10 else None), stats

    def count_falsified(self, assignment):
        a = np.ascontiguousarray(assignment, dtype=np.uint8)
        assert len(a) == self.n_vars + 1
        first = C.c_int()
        n = lib().tsso_cnf_count_falsified(self._h, _p(a, C.c_uint8), C.byref(first))
        return n, first.value

    def propagate(self, assignment):
        """Unit propagation to the fixpoint in synchronous rounds (oracle/capi.cpp tsso_cnf_propagate).
        -> (assignment uint8[n_vars+1], conflict clause index or -1, rounds)"""
        a = np.ascontiguousarray(assignment, dtype=np.uint8).copy()
        assert len(a) == self.n_vars + 1
        conflict, rounds = C.c_int(), C.c_int()
        lib().tsso_cnf_propagate(self._h, _p(a, C.c_uint8), C.byref(conflict), C.byref(rounds))
        return a, conflict.value, rounds.value

    def dimacs(self) -> str:
        lines = [f"p cnf {self.n_vars} {self.n_clauses}"]
        lines += [" ".join(map(str, c)) + " 0" for c in self.clauses()]
        return "\n".join(lines) + "\n"


class Encoding:
    """src/encoder.rs:428-667"""

    def __init__(self, defs, grid):
        self.grid = _grid(grid)
        self.defs = [tuple(d) for d in defs]
        d = _i32(self.defs)
        self._h = C.c_void_p(lib().tsso_encode(_p(self.grid, C.c_uint8), self.grid.shape[1], self.grid.shape[0], _p(d), len(d)))
        K = lib().tsso_encoding_num_dims(self._h)
        dims = np.zeros((K, 2), np.int32)
        lib().tsso_encoding_dims(self._h, _p(dims))
        self.dims = [tuple(map(int, x)) for x in dims]
        tiles = self.grid.size
        self.plat_var = np.zeros((tiles, K), np.int32)
        self.terr_var = np.zeros((tiles, 4), np.int32)
        lib().tsso_encoding_var_maps(self._h, _p(self.plat_var), _p(self.terr_var))

    def __del__(self):
        if lib is not None and self._h:
            lib().tsso_encoding_free(self._h)
            self._h = None

    def cnf(self) -> Cnf:
        return Cnf(lib().tsso_encoding_cnf(self._h))

    def with_limits(self, card_limits=None, weights=None, weight_limit=None) -> Cnf:
        """card_limits / weights: {(w, h): value} keyed by canonical def dims (platform_limits.rs:6-13)"""
        card = _i32([[k[0], k[1], v] for k, v in (card_limits or {}).items()]).reshape(-1, 3)
        wts = _i32([[k[0], k[1], v] for k, v in (weights or {}).items()]).reshape(-1, 3)
        h = lib().tsso_with_limits(self._h, _p(card), len(card), _p(wts), len(wts),
                                   int(weight_limit is not None), C.c_long(weight_limit or 0))
        return Cnf(h)

    def layout_from_assignment(self, assignment):
        a = np.ascontiguousarray(assignment, dtype=np.uint8)
        out = np.zeros((self.grid.size + 1, 5), np.int32)
        n = lib().tsso_layout_from_assignment(self._h, _p(a, C.c_uint8), len(a), _p(out), len(out))
        return [tuple(map(int, p)) for p in out[:n]]

    def assignment_total_weight(self, assignment, weights):
        a = np.ascontiguousarray(assignment, dtype=np.uint8)
        wts = _i32([[k[0], k[1], v] for k, v in weights.items()]).reshape(-1, 3)
        return int(lib().tsso_assignment_total_weight(self._h, _p(a, C.c_uint8), len(a), _p(wts), len(wts)))


# --------------------------------------------------------------------------- layout
@dataclass
class Validation:
    unsupported: np.ndarray  # uint8[h, w]
    overlapping: list
    out_of_bounds: list

    @property
    def is_valid(self):
        return not self.unsupported.any() and not self.overlapping and not self.out_of_bounds


def validate(grid, platforms) -> Validation:
    """src/encoder/platform_layout.rs:85-149.  platforms: [(x, y, def_w, def_h, rotated)]"""
    g = _grid(grid)
    p = _i32(platforms).reshape(-1, 5)
    uns = np.zeros(g.shape, np.uint8)
    flags = np.zeros(max(len(p), 1), np.uint8)
    lib().tsso_validate(_p(g, C.c_uint8), g.shape[1], g.shape[0], _p(p), len(p), _p(uns, C.c_uint8), _p(flags, C.c_uint8))
    plats = [tuple(map(int, x)) for x in p]
    return Validation(uns, [plats[i] for i in range(len(p)) if flags[i] & 1], [plats[i] for i in range(len(p)) if flags[i] & 2])


def trivial_optimization(grid, platforms):
    g = _grid(grid)
    p = _i32(platforms).reshape(-1, 5)
    out = np.zeros((len(p) + 1, 5), np.int32)
    n = lib().tsso_trivial_optimization(_p(g, C.c_uint8), g.shape[1], g.shape[0], _p(p), len(p), _p(out), len(out))
    return [tuple(map(int, x)) for x in out[:n]]


def total_weight(platforms, weights):
    p = _i32(platforms).reshape(-1, 5)
    wts = _i32([[k[0], k[1], v] for k, v in weights.items()]).reshape(-1, 3)
    return int(lib().tsso_total_weight(_p(p), len(p), _p(wts), len(wts)))


def validate_sites_batch(grid, sites, threads=1, flat=False):
    """sites: uint8[n, h, w] 1x1 support masks -> (uncovered int32[n], count int32[n], seconds).
    flat=False: structure-faithful restatement (sets/maps like the reference); flat=True: plain-C flat-array port."""
    g = _grid(grid)
    s = np.ascontiguousarray(sites, dtype=np.uint8).reshape(-1, g.shape[0], g.shape[1])
    unc = np.zeros(len(s), np.int32)
    cnt = np.zeros(len(s), np.int32)
    fn = lib().tsso_validate_sites_batch_flat if flat else lib().tsso_validate_sites_batch
    fn.restype = C.c_double
    sec = fn(_p(g, C.c_uint8), g.shape[1], g.shape[0], _p(s, C.c_uint8), C.c_long(len(s)),
                                          threads, _p(unc), _p(cnt))
    return unc, cnt, sec


# --------------------------------------------------------------------------- solver_loop
def solver_loop(grid, defs, initial_limit=None, conflict_budget=-1):
    """crates/repl/src/main.rs:280-366 -> dict(steps=[...], best=[platforms], proved_optimal)"""
    g = _grid(grid)
    d = _i32(defs)
    steps = np.zeros((4096, 5), np.int64)
    secs = np.zeros(4096, np.float64)
    plats = np.zeros((g.size + 1, 5), np.int32)
    n_plats, proved = C.c_int(), C.c_int()
    n = lib().tsso_solver_loop(_p(g, C.c_uint8), g.shape[1], g.shape[0], _p(d), len(d),
                               C.c_long(-1 if initial_limit is None else initial_limit), C.c_long(conflict_budget), None,
                               _p(steps, C.c_long), len(steps), _p(secs, C.c_double), _p(plats), len(plats),
                               C.byref(n_plats), C.byref(proved))
    return dict(
        steps=[dict(bound=int(s[0]), result=int(s[1]), count=int(s[2]), valid=bool(s[3]), conflicts=int(s[4]), seconds=float(secs[i]))
               for i, s in enumerate(steps[:n])],
        best=[tuple(map(int, p)) for p in plats[: n_plats.value]],
        proved_optimal=bool(proved.value),
    )


# --------------------------------------------------------------------------- SLS model (oracle/sls_model.cpp)
def sls_model(grid, n_chains, epochs, seed=0, chain_offset=0, noise_pct=20, share_bound=True, init_S=None):
    """Replays kernel (b)'s published step rule on the CPU.  epochs: [(steps, bound, target)].
    -> dict(S uint8[n,32,32], bestS, k, best, step, scored, steps)"""
    g = _grid(grid)
    split = []   # spec: an epoch is at most 32768 steps (the 16-bit tabu stamps never wrap inside one); longer runs are consecutive epochs
    for steps_, bound_, target_ in epochs:
        while steps_ > 0:
            split.append((min(steps_, 32768), bound_, target_))
            steps_ -= 32768
    ep = np.ascontiguousarray(split, dtype=np.int64).reshape(-1, 3)
    init = None if init_S is None else np.ascontiguousarray(init_S, np.uint8).reshape(n_chains, 32, 32)
    S = np.zeros((n_chains, 32, 32), np.uint8)
    bestS = np.zeros((n_chains, 32, 32), np.uint8)
    k = np.zeros(n_chains, np.int32)
    best = np.zeros(n_chains, np.int32)
    step = np.zeros(n_chains, np.uint32)
    scored = np.zeros(n_chains, np.uint64)
    steps = np.zeros(n_chains, np.uint64)
    rc = lib().tsso_sls_model(_p(g, C.c_uint8), g.shape[1], g.shape[0], n_chains, C.c_uint32(chain_offset), C.c_uint64(seed), noise_pct,
                              _p(ep, C.c_longlong), len(ep), int(share_bound), _p(init, C.c_uint8) if init is not None else None, _p(S, C.c_uint8), _p(bestS, C.c_uint8), _p(k), _p(best),
                              _p(step, C.c_uint32), _p(scored, C.c_uint64), _p(steps, C.c_uint64))
    assert rc == 0
    return dict(S=S, bestS=bestS, k=k, best=best, step=step, scored=scored, steps=steps)


def sls_flat(grid, n_chains, epochs, seed=0, chain_offset=0, noise_pct=20, share_bound=True, init_S=None, threads=1, want_layouts=True):
    """The same step rule as sls_model through the flat-array CPU port (oracle/sls_flat.cpp), chains spread over `threads`
    host threads.  -> sls_model's dict plus flips (supports added + removed per chain) and seconds (wall time of the epochs)."""
    g = _grid(grid)
    split = []
    for steps_, bound_, target_ in epochs:
        while steps_ > 0:
            split.append((min(steps_, 32768), bound_, target_))
            steps_ -= 32768
    ep = np.ascontiguousarray(split, dtype=np.int64).reshape(-1, 3)
    init = None if init_S is None else np.ascontiguousarray(init_S, np.uint8).reshape(n_chains, 32, 32)
    S = np.zeros((n_chains, 32, 32), np.uint8) if want_layouts else None
    bestS = np.zeros((n_chains, 32, 32), np.uint8) if want_layouts else None
    k = np.zeros(n_chains, np.int32)
    best = np.zeros(n_chains, np.int32)
    step = np.zeros(n_chains, np.uint32)
    scored, steps, flips = np.zeros(n_chains, np.uint64), np.zeros(n_chains, np.uint64), np.zeros(n_chains, np.uint64)
    sec = C.c_double()
    ep_sec, ep_flips = np.zeros(len(ep), np.float64), np.zeros(len(ep), np.uint64)
    rc = lib().tsso_sls_flat(_p(g, C.c_uint8), g.shape[1], g.shape[0], n_chains, C.c_uint32(chain_offset), C.c_uint64(seed), noise_pct,
                             _p(ep, C.c_longlong), len(ep), int(share_bound), _p(init, C.c_uint8) if init is not None else None, int(threads),
                             _p(S, C.c_uint8) if want_layouts else None, _p(bestS, C.c_uint8) if want_layouts else None, _p(k), _p(best),
                             _p(step, C.c_uint32), _p(scored, C.c_uint64), _p(steps, C.c_uint64), _p(flips, C.c_uint64), C.byref(sec),
                             _p(ep_sec, C.c_double), _p(ep_flips, C.c_uint64))
    assert rc == 0
    return dict(S=S, bestS=bestS, k=k, best=best, step=step, scored=scored, steps=steps, flips=flips, seconds=sec.value,
                epoch_seconds=ep_sec, epoch_flips=ep_flips)


def lns_model(grid, seeds, phases, phase_steps, seed=0, chain_offset=0, noise_pct=20, flat=False, threads=1, stats=None, ranks=None):
    """Scalar replay of the window decomposition for grids larger than 32x32 (timberborn_support_solver_b200/csrc/lns.cu): the
    layout starts as "a support under every ceiling tile"; phase p tiles the grid with 32x32 windows at offset OFF[p & 3], freezes
    the supports outside the windows' 26x26 cores, and in every window `seeds` chains of the WINDOW-mode step rule look for a
    complete window layout with fewer core supports; the best chain (lowest index on ties) rewrites the core.
    flat: the windows' chains through the flat-array port (oracle/sls_flat.cpp, the fast CPU implementation: same results), one
    window per worker thread; stats (a dict) then receives the flips and the seconds spent in the chains.
    ranks: [(chain_offset, noise_pct), ...] — the multi-GPU portfolio (csrc/lns.cu window_keys_kernel / contribute_windows_kernel): every
    rank searches every window with its own chains; per window the rank with the fewest core supports wins (lowest rank on ties).
    -> list of (layout uint8[h, w], count) after every phase."""
    C_ = _grid(grid).astype(np.uint8)
    h, w = C_.shape
    S = C_.copy()
    CORE_LO, CORE_HI = 3, 29
    OFF = [(0, 0), (-16, -16), (0, -16), (-16, 0)]
    out = []
    L = lib()
    for phase in range(phases):
        ox, oy = OFF[phase & 3]
        corex = np.array([CORE_LO <= ((x - ox) & 31) < CORE_HI for x in range(w)])
        corey = np.array([CORE_LO <= ((y - oy) & 31) < CORE_HI for y in range(h)])
        core = np.outer(corey, corex)
        F = S & ~core & C_                                   # frozen supports (under ceiling: only those support anything)
        cov = F.copy()
        for _ in range(3):                                   # exact geodesic cover of the frozen supports
            nb = cov.copy()
            nb[:, 1:] |= cov[:, :-1]; nb[:, :-1] |= cov[:, 1:]; nb[1:, :] |= cov[:-1, :]; nb[:-1, :] |= cov[1:, :]
            cov = nb & C_
        nwx, nwy = (w - ox + 31) // 32, (h - oy + 31) // 32
        newS = S.copy()

        def one(win):
            gx0, gy0 = ox + 32 * (win % nwx), oy + 32 * (win // nwx)

            def cut(X):
                W_ = np.zeros((32, 32), np.uint8)
                x0, x1, y0, y1 = max(gx0, 0), min(gx0 + 32, w), max(gy0, 0), min(gy0 + 32, h)
                if x1 > x0 and y1 > y0:
                    W_[y0 - gy0:y1 - gy0, x0 - gx0:x1 - gx0] = X[y0:y1, x0:x1]
                return W_
            c, s_, f = cut(C_), cut(S), cut(cov)
            corew = np.zeros((32, 32), np.uint8)
            corew[CORE_LO:CORE_HI, CORE_LO:CORE_HI] = 1
            score = np.ascontiguousarray((s_ & corew & c).astype(np.uint8))
            need = np.ascontiguousarray((c & (1 - f)).astype(np.uint8))
            c = np.ascontiguousarray(c)
            win_key, win_rows, n_flips = None, None, 0
            for r, (r_offset, r_noise) in enumerate(ranks or [(chain_offset, noise_pct)]):
                bestS = np.zeros((seeds, 32, 32), np.uint8)
                best, k = np.zeros(seeds, np.int32), np.zeros(seeds, np.int32)
                flips = np.zeros(seeds, np.uint64)
                args = (_p(c, C.c_uint8), _p(need, C.c_uint8), CORE_LO, CORE_HI, seeds, C.c_uint32(r_offset + win * seeds), C.c_uint64(seed), r_noise,
                        C.c_longlong(phase_steps), _p(score, C.c_uint8), C.c_uint32(((phase + 1) << 20) & 0xffffffff), _p(bestS, C.c_uint8), _p(best), _p(k))
                if flat:
                    L.tsso_sls_window_flat(*args, _p(flips, C.c_uint64))
                else:
                    L.tsso_sls_window_model(*args)
                winner = int(np.argmin(best))                # lowest chain on ties
                key = int(best[winner]) * 64 + r             # fewest core supports, lowest rank on ties
                n_flips += int(flips.sum())
                if win_key is None or key < win_key:
                    win_key, win_rows = key, bestS[winner] & corew
            return gx0, gy0, win_rows, n_flips

        import time as _time
        t0 = _time.perf_counter()
        if flat and threads > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(threads) as ex:
                results = list(ex.map(one, range(nwx * nwy)))
        else:
            results = [one(win) for win in range(nwx * nwy)]
        if stats is not None:
            stats["seconds"] = stats.get("seconds", 0.0) + _time.perf_counter() - t0
            stats["flips"] = stats.get("flips", 0) + sum(r[3] for r in results)
        for gx0, gy0, rows, _ in results:                    # cores of different windows never overlap: the order does not matter
            x0, x1, y0, y1 = max(gx0 + CORE_LO, 0), min(gx0 + CORE_HI, w), max(gy0 + CORE_LO, 0), min(gy0 + CORE_HI, h)
            if x1 > x0 and y1 > y0:
                newS[y0:y1, x0:x1] = rows[y0 - gy0:y1 - gy0, x0 - gx0:x1 - gx0]
        S = newS
        out.append((S.copy(), int(S.sum())))
    return out


def slsm_model(grid, key_dims, costs, n_chains, epochs, seed=0, chain_offset=0, noise_pct=20, share_bound=True, count_flips=False):
    """Replays the placement search (platform sets beyond {1x1}) on the CPU.  key_dims: [(w, h)] effective dims per key in
    the engine's key order, costs: objective cost per key, epochs: [(steps, bound, target)].
    -> dict(items uint16[n,1024], k, best_items, best_k, best, step, scored_total, steps_total), plus flips_total with
    count_flips (the totals are the engine's tss_stats candidates_scored / sls_steps / sls_flips: flips = platforms added +
    removed).  Without count_flips the dict has the keys callers compare key by key against other replays of the step rule."""
    g = _grid(grid)
    kd = np.ascontiguousarray(key_dims, np.int32).reshape(-1, 2)
    cs = np.ascontiguousarray(costs, np.int32)
    ep = np.ascontiguousarray(epochs, dtype=np.int64).reshape(-1, 3)
    items = np.zeros((n_chains, 1024), np.uint16)
    best_items = np.zeros((n_chains, 1024), np.uint16)
    k, best_k, best = np.zeros(n_chains, np.int32), np.zeros(n_chains, np.int32), np.zeros(n_chains, np.int32)
    step = np.zeros(n_chains, np.uint32)
    totals = np.zeros(3, np.uint64)
    rc = lib().tsso_slsm_model(_p(g, C.c_uint8), g.shape[1], g.shape[0], _p(kd), _p(cs), len(cs), n_chains, C.c_uint32(chain_offset), C.c_uint64(seed),
                               noise_pct, _p(ep, C.c_longlong), len(ep), int(share_bound), _p(items, C.c_uint16), _p(k), _p(best_items, C.c_uint16),
                               _p(best_k), _p(best), _p(step, C.c_uint32), _p(totals, C.c_uint64))
    assert rc == 0
    out = dict(items=items, k=k, best_items=best_items, best_k=best_k, best=best, step=step, scored_total=int(totals[0]), steps_total=int(totals[1]))
    if count_flips:
        out["flips_total"] = int(totals[2])
    return out
