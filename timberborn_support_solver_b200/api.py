"""Host-side mirror of the reference's interface for the feasibility-and-bound path, over the C ABI of libtss.

Names, argument meaning and error behaviour follow the reference lib crate and its two drivers:
  World / WorldGrid / Project           src/world.rs:13-19,96-103, src/lib.rs:15-17
  PlatformDef / Platform                src/platform.rs:11-32,64-118
  Encoding.encode / with_limits / vars  src/encoder.rs:435,615,619
  PlatformLimits                        src/encoder/platform_limits.rs:6-26
  PlatformLayout.*                      src/encoder/platform_layout.rs:26-183  (validate runs on the GPU: kernel (a))
  GpuBoundSolver                        the `Solve + Interrupt + SolveStats` shape the drivers are generic over
                                        (crates/repl/src/solver_runner.rs:8-20, crates/gui/src/solver_backend.rs:69-97)
  solver_loop                           crates/repl/src/main.rs:280-366
Everything that computes goes through libtss (ctypes); nothing here imports oracle/.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Callable, Iterable, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import Dims as _Dims
from ._lib import Platform as _Platform

SAT, UNSAT, INTERRUPTED = "Sat", "Unsat", "Interrupted"  # rustsat SolverResult
KERNEL_AUTO, KERNEL_WARP, KERNEL_HALF_WARP, KERNEL_THREAD, KERNEL_PAIR = 0, 1, 2, 3, 4  # tss.h TSS_KERNEL_*: equivalent SLS kernels
KERNEL_WINDOW_PLACEMENTS = 5  # tss.h: the window-decomposed placement search on grids larger than 32x32


class TssError(RuntimeError):
    def __init__(self, code: int, message: str = ""):
        self.code = code
        super().__init__(f"{_lib.ERROR_NAMES.get(code, code)}: {message}" if message else str(_lib.ERROR_NAMES.get(code, code)))


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


# ------------------------------------------------------------------------------------------------- domain types
@dataclass(frozen=True, order=True)
class PlatformDef:
    """src/platform.rs:11-15; dims are canonical (width <= height as in PLATFORMS_DEFAULT)."""
    width: int
    height: int

    def dims(self):
        return (self.width, self.height)

    def dimensions_str(self) -> str:
        return f"{self.width}x{self.height}"

    def rectangular(self) -> bool:  # platform.rs:51-53
        return self.width != self.height


PLATFORMS_DEFAULT = tuple(PlatformDef(w, h) for w, h in [(1, 1), (1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (3, 3), (5, 5)])


@dataclass(frozen=True, order=True)
class Platform:
    """src/platform.rs:64-70: anchor point (min corner), def, rotated."""
    x: int
    y: int
    definition: PlatformDef
    rotated: bool = False

    def point(self):
        return (self.x, self.y)

    def dims(self):  # platform.rs:111-113
        return (self.definition.height, self.definition.width) if self.rotated else self.definition.dims()

    def _c(self) -> _Platform:
        return _Platform(self.x, self.y, self.definition.width, self.definition.height, int(self.rotated))

    def overlaps(self, other: "Platform") -> bool:  # platform.rs:86-97
        a, b = self._c(), other._c()
        return bool(_lib.load().tss_platform_overlaps(C.byref(a), C.byref(b)))

    @staticmethod
    def _from_c(p: _Platform) -> "Platform":
        return Platform(p.x, p.y, PlatformDef(p.def_w, p.def_h), bool(p.rotated))


def _plat_array(platforms: Sequence[Platform]):
    arr = (_Platform * max(len(platforms), 1))()
    for i, p in enumerate(platforms):
        arr[i] = p._c()
    return arr


def _defs_array(defs: Sequence[PlatformDef]):
    arr = (_Dims * max(len(defs), 1))()
    for i, d in enumerate(defs):
        arr[i] = _Dims(d.width, d.height)
    return arr


class WorldGrid:
    """src/world.rs:19 — Grid<bool>, row-major, index x + y*width (src/math/grid.rs:66-68)."""

    def __init__(self, data):
        self.data = _u8(np.asarray(data) != 0)
        if self.data.ndim != 2 or self.data.size == 0:
            raise ValueError("WorldGrid needs a non-empty 2-D array")

    @property
    def width(self):
        return self.data.shape[1]

    @property
    def height(self):
        return self.data.shape[0]

    def dims(self):
        return (self.width, self.height)

    def get(self, x, y):
        return bool(self.data[y, x]) if 0 <= x < self.width and 0 <= y < self.height else None

    @staticmethod
    def from_toml(text: str) -> "WorldGrid":
        """world.rs:49-79: rows of `X` / space; any other character or an empty array is an error."""
        lib = _lib.load()
        buf = np.zeros(max(len(text), 16), np.uint8)
        w, h, rg = C.c_int32(), C.c_int32(), C.c_int32()
        err = C.create_string_buffer(256)
        rc = lib.tss_world_parse_toml(text.encode(), _ptr(buf, C.c_uint8), buf.size, C.byref(w), C.byref(h), C.byref(rg), err, 256)
        if rc != 0:
            raise TssError(rc, err.value.decode())
        g = WorldGrid(buf[: w.value * h.value].reshape(h.value, w.value))
        g.ragged = bool(rg.value)
        return g

    def to_toml(self) -> str:
        buf = C.create_string_buffer(self.data.size + 16 * self.height + 64)
        n = _lib.load().tss_world_to_toml(_ptr(self.data, C.c_uint8), self.width, self.height, buf, len(buf))
        if n < 0:
            raise TssError(n)
        return buf.value.decode()

    @staticmethod
    def synthetic(w: int, h: int, seed: int = 1, t: int = 0, density: float = 0.7) -> "WorldGrid":
        """SURVEY.md §8(d) generator shared by host, CUDA and tests."""
        g = np.zeros((h, w), np.uint8)
        _lib.load().tss_world_synthetic(w, h, seed, t, int(density * (1 << 24)), _ptr(g, C.c_uint8))
        return WorldGrid(g)


@dataclass
class World:  # src/world.rs:13-16,96-103
    _grid: WorldGrid

    def grid(self) -> WorldGrid:
        return self._grid


@dataclass
class Project:  # src/lib.rs:15-17, crates/repl/src/main.rs:272-278
    world: World

    @staticmethod
    def load(path: str) -> "Project":
        with open(path, "r", encoding="utf-8") as f:
            return Project(World(WorldGrid.from_toml(f.read())))


@dataclass
class PlatformLimits:  # src/encoder/platform_limits.rs:6-13
    card_limits: dict = field(default_factory=dict)   # PlatformDef -> usize
    weights: dict = field(default_factory=dict)       # PlatformDef -> isize
    weight_limit: Optional[int] = None

    @staticmethod
    def new_unweighted(limits: dict) -> "PlatformLimits":
        return PlatformLimits(dict(limits), {}, None)


@dataclass
class Cnf:
    """rustsat Cnf after SatInstance::into_cnf(): CSR clauses, DIMACS-signed literals."""
    n_vars: int
    lits: np.ndarray      # int32
    offsets: np.ndarray   # uint32 [n_clauses + 1]

    @property
    def n_clauses(self):
        return len(self.offsets) - 1

    def clauses(self):
        o = self.offsets
        return [tuple(int(x) for x in self.lits[o[i]: o[i + 1]]) for i in range(self.n_clauses)]


class EncodingVars:
    """src/encoder.rs:175-279 — explicit var maps instead of hash-order numbering."""

    def __init__(self, dims, plat_var, terr_var, width, height):
        self.dims, self.plat_var, self.terr_var, self.width, self.height = dims, plat_var, terr_var, width, height

    def for_dims_at(self, x, y, dims):
        return int(self.plat_var[y * self.width + x, self.dims.index(tuple(dims))])

    def terrain_at(self, x, y):
        t = self.terr_var[y * self.width + x]
        return None if t[0] == 0 else [int(v) for v in t]


class Encoding:
    """src/encoder.rs:428-667."""

    def __init__(self, handle, grid: WorldGrid, defs):
        self._h, self._grid, self.defs = handle, grid, tuple(defs)
        lib = _lib.load()
        nv, nc, nl, nd = C.c_int32(), C.c_int32(), C.c_int64(), C.c_int32()
        lib.tss_encoding_sizes(self._h, C.byref(nv), C.byref(nc), C.byref(nl), C.byref(nd))
        self.n_vars, self.n_clauses, self.n_lits, K = nv.value, nc.value, nl.value, nd.value
        dims = (_Dims * K)()
        lib.tss_encoding_dims(self._h, dims)
        plat = np.zeros((grid.data.size, K), np.int32)
        terr = np.zeros((grid.data.size, 4), np.int32)
        lib.tss_encoding_var_maps(self._h, _ptr(plat, C.c_int32), _ptr(terr, C.c_int32))
        self._vars = EncodingVars([(d.w, d.h) for d in dims], plat, terr, grid.width, grid.height)

    @staticmethod
    def encode(platform_defs: Iterable[PlatformDef], terrain: WorldGrid) -> "Encoding":
        defs = list(platform_defs)
        h = C.c_void_p()
        rc = _lib.load().tss_encoding_create(_ptr(terrain.data, C.c_uint8), terrain.width, terrain.height, _defs_array(defs), len(defs), C.byref(h))
        if rc != 0:
            raise TssError(rc, "Encoding::encode rejected its input (the platform set must contain 1x1; src/encoder.rs:564-566)")
        return Encoding(h, terrain, defs)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None and getattr(_lib, "load", None) is not None:   # (module globals are gone at interpreter shutdown)
            _lib.load().tss_encoding_destroy(self._h)
            self._h = None

    def vars(self) -> EncodingVars:
        return self._vars

    def cnf(self) -> Cnf:
        lits = np.zeros(max(self.n_lits, 1), np.int32)
        offsets = np.zeros(self.n_clauses + 1, np.uint32)
        _lib.load().tss_encoding_cnf(self._h, _ptr(lits, C.c_int32), _ptr(offsets, C.c_uint32))
        return Cnf(self.n_vars, lits[: self.n_lits], offsets)

    def with_limits(self, limits: PlatformLimits) -> Cnf:
        """encoder.rs:619-667 followed by into_cnf() (crates/repl/src/main.rs:292-293)."""
        card = np.array([[d.width, d.height, v] for d, v in limits.card_limits.items()], np.int32).reshape(-1, 3)
        wts = np.array([[d.width, d.height, v] for d, v in limits.weights.items()], np.int32).reshape(-1, 3)
        lib = _lib.load()
        args = (self._h, _ptr(card, C.c_int32), len(card), _ptr(wts, C.c_int32), len(wts), int(limits.weight_limit is not None),
                int(limits.weight_limit or 0))
        nv, nc, nl = C.c_int32(), C.c_int32(), C.c_int64()
        rc = lib.tss_encoding_with_limits(*args, C.byref(nv), C.byref(nc), C.byref(nl), None, None)
        if rc != 0:
            raise TssError(rc)
        lits = np.zeros(max(nl.value, 1), np.int32)
        offsets = np.zeros(nc.value + 1, np.uint32)
        lib.tss_encoding_with_limits(*args, None, None, None, _ptr(lits, C.c_int32), _ptr(offsets, C.c_uint32))
        return Cnf(nv.value, lits[: nl.value], offsets)


@dataclass
class ValidationResult:  # src/encoder/platform_layout.rs:187-191
    unsupported_terrain: set
    overlapping_platforms: set
    out_of_bounds_platforms: set

    def is_valid(self) -> bool:
        return not (self.unsupported_terrain or self.overlapping_platforms or self.out_of_bounds_platforms)


class PlatformLayout:
    """src/encoder/platform_layout.rs:20-183."""

    def __init__(self, platforms: Iterable[Platform] = ()):
        self._platforms = {p.point(): p for p in platforms}

    @staticmethod
    def from_assignment(assignment, encoding: Encoding) -> "PlatformLayout":
        a = _u8(assignment)
        out = (_Platform * (encoding._grid.data.size + 1))()
        n = C.c_int32()
        rc = _lib.load().tss_layout_from_assignment(encoding._h, _ptr(a, C.c_uint8), len(a), out, len(out), C.byref(n))
        if rc != 0:
            raise TssError(rc)
        return PlatformLayout(Platform._from_c(out[i]) for i in range(n.value))

    def platforms(self):
        return self._platforms

    def platform_count(self) -> int:
        return len(self._platforms)

    def platform_stats(self) -> dict:
        out: dict = {}
        for p in self._platforms.values():
            out[p.definition] = out.get(p.definition, 0) + 1
        return out

    def get_platform(self, point):
        return self._platforms.get(tuple(point))

    def validate(self, world: World, engine: "Engine") -> ValidationResult:
        """platform_layout.rs:85-149 — computed by the coverage kernel (a)."""
        return engine.validate(world.grid(), list(self._platforms.values()))

    def run_trivial_optimization(self, world: World) -> None:
        g = world.grid()
        plats = list(self._platforms.values())
        arr = _plat_array(plats)
        n = _lib.load().tss_layout_trivial_optimization(_ptr(g.data, C.c_uint8), g.width, g.height, arr, len(plats))
        if n < 0:
            raise TssError(n)
        self._platforms = {(arr[i].x, arr[i].y): Platform._from_c(arr[i]) for i in range(n)}

    def merge_supports(self, world: World, defs) -> None:
        """A layout of 1x1 supports, re-expressed with the larger platforms of `defs` where supports fit under one footprint
        (host-side; the engine applies it to its window-decomposed search on grids larger than 32x32)."""
        g = world.grid()
        plats = list(self._platforms.values())
        arr = _plat_array(plats)
        defs = list(defs)
        n = _lib.load().tss_layout_merge_supports(_ptr(g.data, C.c_uint8), g.width, g.height, _defs_array(defs), len(defs), arr, len(plats), len(plats))
        if n < 0:
            raise TssError(n)
        self._platforms = {(arr[i].x, arr[i].y): Platform._from_c(arr[i]) for i in range(n)}

    def total_weight(self, weights: dict) -> int:
        plats = list(self._platforms.values())
        wts = np.array([[d.width, d.height, v] for d, v in weights.items()], np.int32).reshape(-1, 3)
        return int(_lib.load().tss_layout_total_weight(_plat_array(plats), len(plats), _ptr(wts, C.c_int32), len(wts)))


# Box-drawing glyph by the directions a platform tile CONNECTS to, index = N<<3 | S<<2 | W<<1 | E
# (crates/repl/src/main.rs:524-549)
_BOX = " ╶╴─╷┌┐┬╵└┘┴│├┤┼"


def render_world(world: World, layout: Optional[PlatformLayout] = None, validation: Optional[ValidationResult] = None, color: bool = False) -> str:
    """The REPL's map printout (crates/repl/src/main.rs:390-480): one glyph + two spaces per tile, one line per grid row.
    Empty = ' ', ceiling = '▒' (yellow when unsupported), 1x1 platform = '☐', larger platforms as an outline of box
    characters (interior blank, straight runs drawn as │ / ─), overlapping platforms red.  Platform tiles outside the
    grid are dropped.  `color` adds the ANSI sequences owo-colors emits (ESC[33m / ESC[31m ... ESC[39m)."""
    g = world.grid()
    h, w = g.height, g.width
    unsupported = validation.unsupported_terrain if validation else set()
    overlapping = validation.overlapping_platforms if validation else set()
    paint = (lambda t, c: f"\x1b[{c}m{t}\x1b[39m") if color else (lambda t, c: t)
    cells = [[" "] * w for _ in range(h)]
    for y in range(h):
        for x in range(w):
            if g.data[y, x]:
                cells[y][x] = paint("▒", 33) if (x, y) in unsupported else "▒"
    for plat in (layout.platforms().values() if layout else ()):
        pw, ph = plat.dims()
        red = plat in overlapping
        for ry in range(ph):
            for rx in range(pw):
                x, y = plat.x + rx, plat.y + ry
                if not (0 <= x < w and 0 <= y < h):
                    continue
                # open = no platform tile of this platform in that direction
                n_open, s_open, w_open, e_open = ry == 0, ry == ph - 1, rx == 0, rx == pw - 1
                if n_open and s_open and w_open and e_open:
                    glyph = "☐"
                else:
                    if not (n_open or s_open or w_open or e_open):      # interior: blank
                        n_open = s_open = w_open = e_open = True
                    elif not (n_open or s_open):                          # vertical run: ignore the sides
                        w_open = e_open = True
                    elif not (w_open or e_open):                          # horizontal run
                        n_open = s_open = True
                    glyph = _BOX[(not n_open) << 3 | (not s_open) << 2 | (not w_open) << 1 | (not e_open)]
                cells[y][x] = paint(glyph, 31) if red else glyph
    return "".join("".join(c + "  " for c in row) + "\n" for row in cells)


# ------------------------------------------------------------------------------------------------- engine
class DeviceCnf:
    def __init__(self, engine: "Engine", cnf: Cnf):
        self.engine, self.cnf = engine, cnf
        self._h = C.c_void_p()
        lits = np.ascontiguousarray(cnf.lits, np.int32)
        offs = np.ascontiguousarray(cnf.offsets, np.uint32)
        engine._check(engine.lib.tss_cnf_upload(engine._h, _ptr(lits, C.c_int32), _ptr(offs, C.c_uint32), cnf.n_clauses, cnf.n_vars, C.byref(self._h)))

    def __del__(self):
        if getattr(self, "_h", None) and self.engine._h:
            self.engine.lib.tss_cnf_destroy(self._h)
            self._h = None

    def check(self, assignments):
        """-> (n_falsified int32[n], first_falsified int32[n])"""
        a = _u8(assignments).reshape(-1, self.cnf.n_vars + 1)
        nf = np.zeros(len(a), np.int32)
        first = np.zeros(len(a), np.int32)
        e = self.engine
        e._check(e.lib.tss_cnf_check(e._h, self._h, _ptr(a, C.c_uint8), len(a), _ptr(nf, C.c_int32), _ptr(first, C.c_int32)))
        return nf, first

    def propagate(self, assignments):
        """Unit propagation to fixpoint -> (assignments uint8[n, n_vars+1], conflict int32[n], rounds)"""
        a = _u8(assignments).reshape(-1, self.cnf.n_vars + 1).copy()
        conflict = np.zeros(len(a), np.int32)
        rounds = C.c_int32()
        e = self.engine
        e._check(e.lib.tss_cnf_propagate(e._h, self._h, _ptr(a, C.c_uint8), len(a), _ptr(conflict, C.c_int32), C.byref(rounds)))
        return a, conflict, rounds.value

    def complete(self, assignment):
        """tss_cnf_complete: ONE partial assignment -> (completed assignment uint8[n_vars + 1], conflict clause or -1, clauses falsified):
        unit propagation, open variables False, clause check — one fused launch when the variables fit a CTA's shared memory."""
        a = _u8(assignment).reshape(self.cnf.n_vars + 1).copy()
        conflict, nf = C.c_int32(-1), C.c_int32(0)
        e = self.engine
        e._check(e.lib.tss_cnf_complete(e._h, self._h, _ptr(a, C.c_uint8), C.byref(conflict), C.byref(nf)))
        return a, conflict.value, nf.value

    def witness(self, encoding: "Encoding", layout: "PlatformLayout"):
        """tss_witness_for_cnf: the layout completed into a model of these clauses (platform + terrain-layer variables from the
        layout, auxiliaries by unit propagation, open variables False, every clause checked — one fused launch, csrc/cnf.cu
        cnf_complete_kernel) -> assignment uint8[n_vars + 1], or None when it is not a model (e.g. the layout exceeds a limit)."""
        plats = list(layout.platforms().values())
        a = np.zeros(self.cnf.n_vars + 1, np.uint8)
        e = self.engine
        rc = e._check(e.lib.tss_witness_for_cnf(e._h, self._h, encoding._h, _plat_array(plats), len(plats), _ptr(a, C.c_uint8)))
        return a if rc == 10 else None


def _card_records(limits: dict) -> np.ndarray:
    return np.array([[d.width, d.height, v] for d, v in limits.items()], np.int32).reshape(-1, 3)


def card_limit_classes(defs, limits: dict):
    """The classes per-type limits constrain, as Encoding::with_limits lowers them (tss_card_limit_classes; host only):
    limits {PlatformDef: limit} -> (key_dims [(w, h)] in the engine's key order, key_mask [int] per key (bit j = class j),
    class_limit [int]).  1x1 and vacuous entries make no class."""
    defs = list(defs)
    card = _card_records(limits)
    mask, lim = (C.c_int32 * 16)(), (C.c_int32 * 16)()
    nk, nc = C.c_int32(), C.c_int32()
    lib = _lib.load()
    rc = lib.tss_card_limit_classes(_defs_array(defs), len(defs), _ptr(card, C.c_int32) if len(card) else None, len(card), mask, lim, C.byref(nk), C.byref(nc))
    if rc < 0:
        raise TssError(rc, "tss_card_limit_classes")
    keys = []
    for d in defs:
        for k in ((d.width, d.height), (d.height, d.width)):
            if k not in keys:
                keys.append(k)
    assert len(keys) == nk.value
    return keys, [int(mask[i]) for i in range(nk.value)], [int(lim[j]) for j in range(nc.value)]


class Search:
    """A device-resident SLS portfolio on one terrain (kernel (b))."""

    def __init__(self, engine: "Engine", grid: WorldGrid, defs=PLATFORMS_DEFAULT[:1], seed=0, n_chains=0, chain_offset=0, noise_pct=-1, kernel=0):
        """kernel: KERNEL_AUTO / KERNEL_WARP / KERNEL_HALF_WARP / KERNEL_THREAD / KERNEL_PAIR (tss.h TSS_KERNEL_*): equivalent SLS kernels
        (KERNEL_PAIR: one chain per thread with two grid rows per word, grids of at most 16x16).  KERNEL_WINDOW_PLACEMENTS: the
        window-decomposed placement search on grids larger than 32x32 with platforms beyond 1x1 (n_chains = chains per window); each
        run() is a phase that can only improve the global layout, best_layout() returns it (before the first run: the greedy cover)."""
        self.engine, self.grid = engine, grid
        self._h = C.c_void_p()
        params = _lib.SearchParams(seed, n_chains, chain_offset, noise_pct, kernel)
        defs = list(defs)
        engine._check(engine.lib.tss_search_create(engine._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _defs_array(defs), len(defs),
                                                   C.byref(params), C.byref(self._h)))
        self.n_chains = engine.lib.tss_search_n_chains(self._h)

    def close(self):
        if getattr(self, "_h", None) and self.engine._h:
            self.engine.lib.tss_search_destroy(self._h)
            self._h = None

    __del__ = close

    def kernel_variant(self) -> int:
        """TSS_KERNEL_* the engine runs this portfolio with (what auto resolved to)"""
        return int(self.engine.lib.tss_search_kernel(self._h))

    def run(self, steps: int, target_count: int = 0):
        """One epoch: `steps` SLS steps per chain, asynchronous on the engine stream."""
        self.engine._check(self.engine.lib.tss_search_run(self._h, steps, target_count))

    def best_count(self) -> Optional[int]:
        c = C.c_int32()
        self.engine._check(self.engine.lib.tss_search_best_count(self._h, C.byref(c)))
        return None if c.value < 0 else c.value

    def set_bound(self, count: int):
        self.engine._check(self.engine.lib.tss_search_set_bound(self._h, count))

    def global_best(self) -> Optional[int]:
        """The bound the next epoch searches below (min over this search, outside bounds and — with a communicator on the
        engine — every rank's search)."""
        c = C.c_int32()
        self.engine._check(self.engine.lib.tss_search_global_best(self._h, C.byref(c)))
        return None if c.value < 0 else c.value

    def read_chains(self) -> dict:
        """Per-chain state after the last epoch (parity tests replay it on the CPU model)."""
        n = self.n_chains
        S, bestS = np.zeros((n, 32), np.uint32), np.zeros((n, 32), np.uint32)
        k, best = np.zeros(n, np.int32), np.zeros(n, np.int32)
        step, scored = np.zeros(n, np.uint32), np.zeros(n, np.uint64)
        self.engine._check(self.engine.lib.tss_search_read_chains(self._h, _ptr(S, C.c_uint32), _ptr(bestS, C.c_uint32), _ptr(k, C.c_int32),
                                                                   _ptr(best, C.c_int32), _ptr(step, C.c_uint32), _ptr(scored, C.c_uint64)))
        return dict(S=S, bestS=bestS, k=k, best=best, step=step, scored=scored)

    def set_weights(self, weights: dict):
        """GUI objective (crates/gui/src/app.rs:53-62): {PlatformDef: weight}; the search then minimises total_weight."""
        wts = np.array([[d.width, d.height, v] for d, v in weights.items()], np.int32).reshape(-1, 3)
        self.engine._check(self.engine.lib.tss_search_set_weights(self._h, _ptr(wts, C.c_int32), len(wts)))

    def set_card_limits(self, limits: dict):
        """Per-type platform limits (`solve -l k:v`, PlatformLimits.card_limits without 1x1): {PlatformDef: limit}.  Additions that
        would take a limit's class (card_limit_classes) beyond it are no candidates, so every layout of every chain keeps every
        limit.  Call before the first run(); TssError for a 1x1 entry or a negative limit, and for a limit that is not vacuous on
        anything but the placement search on a grid up to 32x32."""
        card = _card_records(limits)
        self.engine._check(self.engine.lib.tss_search_set_card_limits(self._h, _ptr(card, C.c_int32) if len(card) else None, len(card)))

    def read_placements(self) -> dict:
        """Per-chain state of the placement search (platform sets beyond {1x1}) after the last epoch."""
        n = self.n_chains
        items, best_items = np.zeros((n, 1024), np.uint16), np.zeros((n, 1024), np.uint16)
        k, best_k, best = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32)
        step = np.zeros(n, np.uint32)
        kd = (_Dims * 16)()
        nk = C.c_int32()
        self.engine._check(self.engine.lib.tss_search_read_placements(self._h, _ptr(items, C.c_uint16), _ptr(k, C.c_int32), _ptr(best_items, C.c_uint16),
                                                                       _ptr(best_k, C.c_int32), _ptr(best, C.c_int32), _ptr(step, C.c_uint32), kd, C.byref(nk)))
        return dict(items=items, k=k, best_items=best_items, best_k=best_k, best=best, step=step, key_dims=[(kd[i].w, kd[i].h) for i in range(nk.value)])

    def write_chains(self, S):
        """Warm start: S uint32[n_chains, 32] support rows become every chain's current layout."""
        S = np.ascontiguousarray(S, np.uint32)
        assert S.shape == (self.n_chains, 32)
        self.engine._check(self.engine.lib.tss_search_write_chains(self._h, _ptr(S, C.c_uint32)))

    def best_layout(self) -> PlatformLayout:
        out = (_Platform * (self.grid.data.size + 1))()
        n = C.c_int32()
        self.engine._check(self.engine.lib.tss_search_best_layout(self._h, out, len(out), C.byref(n)))
        return PlatformLayout(Platform._from_c(out[i]) for i in range(n.value))


class Engine:
    """One tss_engine: a GPU, a stream, scratch memory, an interrupt flag."""

    def __init__(self, device: int = -1):
        self.lib = _lib.load()
        self._h = C.c_void_p()
        rc = self.lib.tss_engine_create(device, C.byref(self._h))
        if rc != 0:
            self._h = None
            raise TssError(rc, "no usable CUDA device (the GPU path has no CPU fallback)")

    def close(self):
        if getattr(self, "_h", None):
            self.lib.tss_engine_destroy(self._h)
            self._h = None

    __del__ = close

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise TssError(rc, self.lib.tss_last_error(self._h).decode())
        return rc

    # ---- multi-GPU portfolio (one process per GPU; the host only carries the 128-byte NCCL id between ranks)
    def comm_unique_id(self) -> bytes:
        buf = np.zeros(128, np.uint8)
        self._check(self.lib.tss_comm_unique_id(self._h, _ptr(buf, C.c_uint8)))
        return buf.tobytes()

    def comm_init(self, unique_id: bytes, rank: int, world: int):
        buf = np.frombuffer(unique_id, np.uint8).copy()
        assert buf.size == 128
        self._check(self.lib.tss_comm_init(self._h, _ptr(buf, C.c_uint8), rank, world))

    def comm_world(self) -> int:
        return self.lib.tss_comm_world(self._h)

    def set_stream(self, cuda_stream: int):
        self._check(self.lib.tss_engine_set_stream(self._h, C.c_void_p(cuda_stream)))

    def interrupt(self):
        self.lib.tss_interrupt(self._h)

    def clear_interrupt(self):
        self.lib.tss_clear_interrupt(self._h)

    def stats(self) -> dict:
        s = _lib.Stats()
        self.lib.tss_get_stats(self._h, C.byref(s))
        return {k: getattr(s, k) for k, _ in _lib.Stats._fields_}

    def device_info(self) -> dict:
        name = C.create_string_buffer(128)
        sm, khz = C.c_int(), C.c_int()
        self.lib.tss_device_info(self._h, name, 128, C.byref(sm), C.byref(khz))
        return dict(name=name.value.decode(), sm_count=sm.value, clock_khz=khz.value)

    # ---- kernel (a)
    def validate(self, grid: WorldGrid, platforms: Sequence[Platform]) -> ValidationResult:
        uns = np.zeros((grid.height, grid.width), np.uint8)
        flags = np.zeros(max(len(platforms), 1), np.uint8)
        self._check(self.lib.tss_validate(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _plat_array(platforms), len(platforms),
                                          _ptr(uns, C.c_uint8), _ptr(flags, C.c_uint8)))
        ys, xs = np.nonzero(uns)
        return ValidationResult({(int(x), int(y)) for x, y in zip(xs, ys)},
                                {p for p, f in zip(platforms, flags) if f & 1}, {p for p, f in zip(platforms, flags) if f & 2})

    def eval_sites(self, grid: WorldGrid, sites):
        """sites: uint8[n, h, w] -> (uncovered int32[n], count int32[n])"""
        s = _u8(sites).reshape(-1, grid.height, grid.width)
        unc, cnt = np.zeros(len(s), np.int32), np.zeros(len(s), np.int32)
        self._check(self.lib.tss_eval_sites(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _ptr(s, C.c_uint8), len(s),
                                            _ptr(unc, C.c_int32), _ptr(cnt, C.c_int32)))
        return unc, cnt

    def eval_packed(self, grid_rows, w: int, h: int, layouts):
        g = np.ascontiguousarray(grid_rows, np.uint32)
        l = np.ascontiguousarray(layouts, np.uint32).reshape(-1, g.size)
        unc, cnt = np.zeros(len(l), np.int32), np.zeros(len(l), np.int32)
        self._check(self.lib.tss_eval_packed(self._h, _ptr(g, C.c_uint32), w, h, _ptr(l, C.c_uint32), len(l), _ptr(unc, C.c_int32), _ptr(cnt, C.c_int32)))
        return unc, cnt

    def eval_compact_dev(self, grid_dev_ptr: int, w: int, h: int, layouts_dev_ptr: int, n: int, out_dev_ptr: int, per_layout_terrain=False):
        self._check(self.lib.tss_eval_compact_dev(self._h, C.c_void_p(grid_dev_ptr), w, h, C.c_void_p(layouts_dev_ptr), n, int(per_layout_terrain),
                                                  C.c_void_p(out_dev_ptr)))

    def eval_platforms(self, grid: WorldGrid, layouts: Sequence[Sequence[Platform]]):
        """-> int32[n, 4] = (unsupported tiles, platforms, overlapping platforms, out-of-bounds platforms)"""
        flat = [p for l in layouts for p in l]
        offsets = np.zeros(len(layouts) + 1, np.uint32)
        offsets[1:] = np.cumsum([len(l) for l in layouts])
        out = np.zeros((len(layouts), 4), np.int32)
        self._check(self.lib.tss_eval_platforms(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _plat_array(flat),
                                                _ptr(offsets, C.c_uint32), len(layouts), _ptr(out, C.c_int32)))
        return out

    def layout_to_assignment(self, encoding: Encoding, layout: PlatformLayout) -> np.ndarray:
        plats = list(layout.platforms().values())
        a = np.zeros(encoding.n_vars + 1, np.uint8)
        self._check(self.lib.tss_layout_to_assignment(self._h, encoding._h, _plat_array(plats), len(plats), _ptr(a, C.c_uint8)))
        return a

    # ---- kernel (c)
    def upload_cnf(self, cnf: Cnf) -> DeviceCnf:
        return DeviceCnf(self, cnf)

    # ---- kernel (b)
    def search(self, grid: WorldGrid, defs=PLATFORMS_DEFAULT[:1], **kw) -> Search:
        """A device-resident SLS portfolio; kw: seed, n_chains, chain_offset, noise_pct, kernel (KERNEL_AUTO, or one of KERNEL_WARP /
        KERNEL_HALF_WARP / KERNEL_THREAD / KERNEL_PAIR to pin a variant, or KERNEL_WINDOW_PLACEMENTS for the placement search on
        grids larger than 32x32; a kernel that does not fit the grid or platform set raises TssError)."""
        return Search(self, grid, defs, **kw)

    def solve_upper_bound(self, grid: WorldGrid, defs=PLATFORMS_DEFAULT[:1], card_limit: Optional[int] = None, seed=0, budget_ms=0, max_steps=0):
        """-> (SAT | INTERRUPTED, PlatformLayout | None).  Never UNSAT: the GPU proves nothing."""
        defs = list(defs)
        out = (_Platform * (grid.data.size + 1))()
        n = C.c_int32()
        rc = self._check(self.lib.tss_solve_upper_bound(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _defs_array(defs), len(defs),
                                                        -1 if card_limit is None else card_limit, seed, budget_ms, max_steps, out, len(out), C.byref(n)))
        if rc == _lib.TSS_SAT:
            return SAT, PlatformLayout(Platform._from_c(out[i]) for i in range(n.value))
        return INTERRUPTED, None

    def solve_min_weight(self, grid: WorldGrid, defs, weights: dict, weight_limit: Optional[int] = None, seed=0, budget_ms=0, max_steps=0):
        """GUI objective (crates/gui/src/app.rs:235-245): -> (SAT | INTERRUPTED, PlatformLayout | None, total weight | None)."""
        defs = list(defs)
        wts = np.array([[d.width, d.height, v] for d, v in weights.items()], np.int32).reshape(-1, 3)
        out = (_Platform * (grid.data.size + 1))()
        n, wt = C.c_int32(), C.c_int64()
        rc = self._check(self.lib.tss_solve_min_weight(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _defs_array(defs), len(defs),
                                                       _ptr(wts, C.c_int32), len(wts), -1 if weight_limit is None else weight_limit, seed, budget_ms,
                                                       max_steps, out, len(out), C.byref(n), C.byref(wt)))
        if rc == _lib.TSS_SAT:
            return SAT, PlatformLayout(Platform._from_c(out[i]) for i in range(n.value)), wt.value
        return INTERRUPTED, None, None

    def solve_with_limits(self, grid: WorldGrid, defs, limits: PlatformLimits, seed=0, budget_ms=0, max_steps=0):
        """The PlatformLimits-shaped solve (tss_solve_with_limits): card_limits including the platform count (1x1) and per-type
        limits; with weights the objective is the total weight, bounded by weight_limit (weights and a 1x1 limit together raise
        TssError).  Budgets as solve_upper_bound.  -> (SAT | INTERRUPTED, PlatformLayout | None, objective | None)."""
        defs = list(defs)
        card = _card_records(limits.card_limits)
        wts = _card_records(limits.weights)
        out = (_Platform * (grid.data.size + 1))()
        n, obj = C.c_int32(), C.c_int64()
        wl = -1 if limits.weight_limit is None else limits.weight_limit
        rc = self._check(self.lib.tss_solve_with_limits(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _defs_array(defs), len(defs),
                                                        _ptr(card, C.c_int32) if len(card) else None, len(card), _ptr(wts, C.c_int32) if len(wts) else None,
                                                        len(wts), wl, seed, budget_ms, max_steps, out, len(out), C.byref(n), C.byref(obj)))
        if rc == _lib.TSS_SAT:
            return SAT, PlatformLayout(Platform._from_c(out[i]) for i in range(n.value)), obj.value
        return INTERRUPTED, None, None

    def lower_bound(self, grid: WorldGrid, defs=PLATFORMS_DEFAULT[:1], seed=0, restarts=0):
        """Packing lower bound (tss_lower_bound): -> list of (x, y) ceiling tiles no two of which one platform of `defs` can
        support; its length bounds the platform count of every complete layout from below."""
        defs = list(defs)
        out = np.zeros((grid.data.size + 1, 2), np.int32)
        n = C.c_int32()
        self._check(self.lib.tss_lower_bound(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _defs_array(defs), len(defs), seed, restarts,
                                             _ptr(out, C.c_int32), len(out), C.byref(n)))
        return [(int(x), int(y)) for x, y in out[: n.value]]

    def lower_bound_lp(self, grid: WorldGrid, defs=PLATFORMS_DEFAULT[:1], max_pivots=0, weights: Optional[dict] = None, target=0):
        """Fractional packing lower bound (tss_lower_bound_lp), certified in integers: on the platform count, or with `weights`
        ({PlatformDef: weight}, the PlatformLimits.weights map) on PlatformLayout::total_weight.  target > 0: the simplex stops as
        soon as the bound reaches it (every iterate is feasible; enough for "is there nothing within target - 1?").
        On grids larger than 32x32 (up to 256x256; at most 16 dims keys, each at most 6x6) a first-order method replaces the
        simplex under the same certificate: `max_pivots` caps its iterations (0: 3 000) and the result's `pivots` counts them,
        `target` is checked on the certified bound every 250 iterations, and `optimal` is always False.
        -> dict(bound, weights int32[h, w], total, max_load, pivots, optimal, constraints)."""
        defs = list(defs)
        wts = np.zeros((grid.height, grid.width), np.int32)
        total, max_load, bound = C.c_int64(), C.c_int64(), C.c_int64()
        info = (C.c_int32 * 3)()
        rec = np.array([[d.width, d.height, v] for d, v in (weights or {}).items()], np.int32).reshape(-1, 3)
        self._check(self.lib.tss_lower_bound_lp(self._h, _ptr(grid.data, C.c_uint8), grid.width, grid.height, _defs_array(defs), len(defs),
                                                _ptr(rec, C.c_int32) if len(rec) else None, len(rec), max_pivots, int(target),
                                                _ptr(wts, C.c_int32), C.byref(total), C.byref(max_load), C.byref(bound), info))
        return dict(bound=bound.value, weights=wts, total=total.value, max_load=max_load.value, pivots=info[0], optimal=bool(info[1]), constraints=info[2])

    def solve_batch(self, grids, seed=0, steps=2048, want_layouts=False, chains_per_terrain=0):
        """grids: uint8[n, h, w] -> counts int32[n] (and packed support rows uint32[n, h] if asked)"""
        g = _u8(grids)
        n, h, w = g.shape
        counts = np.zeros(n, np.int32)
        layouts = np.zeros((n, h), np.uint32) if want_layouts else None
        self._check(self.lib.tss_solve_batch(self._h, _ptr(g, C.c_uint8), w, h, n, seed, steps, chains_per_terrain, _ptr(counts, C.c_int32),
                                             _ptr(layouts, C.c_uint32) if want_layouts else None))
        return (counts, layouts) if want_layouts else counts

    def measure_peaks(self) -> dict:
        out = (C.c_double * 8)()
        self._check(self.lib.tss_measure_peaks(self._h, out, 8))
        return dict(lop3_gops=out[0], popc_gops=out[1], shfl_gops=out[2], smem_gbs=out[3], sm_mhz=out[4])


# ------------------------------------------------------------------------------------------------- solver shape
class GpuBoundSolver:
    """The `Solve + Interrupt + SolveStats (+ Default)` shape of rustsat solvers as the drivers use it
    (crates/repl/src/solver_runner.rs:8-20, crates/gui/src/solver_backend.rs:69-97), answered by the GPU engine:
    solve() returns SAT with a CNF-verified witness when a layout within the instance's bound exists in the budget,
    INTERRUPTED (unknown) otherwise — never UNSAT, only the exact solver proves that (see INTEGRATION.md)."""

    def __init__(self, engine: Engine, encoding: Encoding, limits: PlatformLimits, seed=0, budget_ms=50, max_steps=0):
        self.engine, self.encoding, self.limits = engine, encoding, limits
        self.seed, self.budget_ms, self.max_steps = seed, budget_ms, max_steps
        self._cnf: Optional[Cnf] = None
        self._dev: Optional[DeviceCnf] = None
        self._solution = None
        self._layout = None

    def add_cnf(self, cnf: Cnf):  # Solve::add_cnf
        self._cnf = cnf
        self._dev = self.engine.upload_cnf(cnf)

    def interrupter(self) -> Callable[[], None]:  # Interrupt::interrupter
        return self.engine.interrupt

    def solve(self) -> str:  # Solve::solve
        """SAT with a CNF-verified witness, or INTERRUPTED = "the GPU could not answer within its budget" (which is also what a
        real interrupt returns).  The search is steered by the 1x1 card limit (= the platform count, what the REPL tightens,
        main.rs:346) or by the weight limit (the GUI's objective, app.rs:235-245), and by limits on other platform types
        (`solve -l k:v`) on grids up to 32x32; elsewhere such instances go to the exact solver."""
        one = PlatformDef(1, 1)
        bound = self.limits.card_limits.get(one)
        self.engine.clear_interrupt()      # the flag is sticky by design (InterruptSolver::interrupt may fire before solve starts a kernel): one solve, one flag
        weighted = bool(self.limits.weights) and (self.limits.weight_limit is not None or bound is None)
        if any(d != one for d in self.limits.card_limits):
            g = self.encoding._grid
            if g.width > 32 or g.height > 32 or (weighted and bound is not None):
                return INTERRUPTED         # limits the search cannot steer by here: leave the instance to the exact solver
            lim = self.limits if weighted else PlatformLimits(dict(self.limits.card_limits), {}, None)
            res, layout, _ = self.engine.solve_with_limits(g, self.encoding.defs, lim, self.seed, self.budget_ms, self.max_steps)
        elif weighted:
            # the GUI's instances: weights always, a weight limit from the second iteration on (app.rs:235-245)
            res, layout, _ = self.engine.solve_min_weight(self.encoding._grid, self.encoding.defs, self.limits.weights, self.limits.weight_limit,
                                                          self.seed, self.budget_ms, self.max_steps)
        else:
            res, layout = self.engine.solve_upper_bound(self.encoding._grid, self.encoding.defs, bound, self.seed, self.budget_ms, self.max_steps)
        if res != SAT:
            return INTERRUPTED
        if self._cnf is not None:  # witness against the very clauses the exact solver would get (kernel (c)), one fused launch
            a = self._dev.witness(self.encoding, layout)
            if a is None:
                return INTERRUPTED
        else:
            a = self.engine.layout_to_assignment(self.encoding, layout)
        self._solution, self._layout = a, layout
        return SAT

    def full_solution(self):  # Solve::full_solution
        if self._solution is None:
            raise RuntimeError("no solution: solve() did not return Sat")
        return self._solution

    def stats(self) -> dict:  # SolveStats::stats
        return self.engine.stats()


def solver_loop(project: Project, encoding: Encoding, limits: PlatformLimits, engine: Engine, exact_solver=None, seed=0, budget_ms=None,
                on_solution=None, use_lower_bound=True):
    """crates/repl/src/main.rs:280-366 with the GPU engine as the SAT side and an optional exact solver
    (`exact_solver(cnf) -> (SAT|UNSAT|INTERRUPTED, assignment)`, Glucose in the reference) for the proof.

    budget_ms=None (default): every iteration is ONE SAT-like call (first layout within the bound) whose give-up point
    adapts to the run — 32x the steps the previous successful call needed, at least 1024 per chain — so the iteration the
    GPU cannot answer (one below the optimum) costs milliseconds before the prover takes over, not the engine's default
    2^18 steps.  budget_ms=0 keeps that default effort; budget_ms > 0 improves for that long in every iteration.

    use_lower_bound: ask the engine for its packing lower bound first (tss_lower_bound); when the count reaches it the loop
    ends with `proved_optimal` and no exact-solver call.

    Returns dict(best=PlatformLayout|None, proved_optimal=bool, steps=[...], lower_bound=int|None)."""
    one = PlatformDef(1, 1)
    limits = PlatformLimits(dict(limits.card_limits), dict(limits.weights), limits.weight_limit)
    steps, best, proved = [], None, False
    give_up = 1024
    engine.clear_interrupt()
    # lower bounds (not in the reference): once the count meets one — or the next bound falls below it — the loop is finished and
    # nothing is left for the exact solver to prove.  Only when the count is the sole limit (the REPL's case).  The integral
    # packing (tss_lower_bound, ~0.1 ms) is computed up front; the fractional bound (tss_lower_bound_lp, a simplex solve: tens of
    # ms on a 21x16 terrain) only when the GPU has found nothing below a count the packing does not already certify.
    lower, lp_done = None, False
    g = encoding._grid
    only_count = not limits.weights and limits.weight_limit is None and all(d == one for d in limits.card_limits)
    use_lower_bound = use_lower_bound and only_count and g.width <= 32 and g.height <= 32
    if use_lower_bound:
        try:
            lower = len(engine.lower_bound(g, encoding.defs, seed=seed))
        except TssError as err:             # a platform set the bound kernels do not take (more than 16 dims keys): carry on without bounds
            if err.code != _lib.TSS_E_UNSUPPORTED:
                raise
            use_lower_bound = False
    while True:
        bound_now = limits.card_limits.get(one)
        if lower is not None and best is not None and bound_now is not None and bound_now < lower:
            steps.append(dict(bound=bound_now, result=UNSAT, source="lower bound"))
            proved = True
            break
        cnf = encoding.with_limits(limits)                      # main.rs:292-293
        # while the fractional bound is still to be computed the search first gets an eighth of its give-up budget (the limits
        # nothing satisfies are where a long search is wasted), the whole budget only if the bound does not refute the limit:
        # the same schedule as tss_solve_instance (csrc/instance.cpp)
        lp_pending = use_lower_bound and not lp_done and best is not None
        first = max(128, give_up // 8) if (budget_ms is None and lp_pending) else give_up
        if budget_ms is None:
            solver = GpuBoundSolver(engine, encoding, limits, seed=seed, budget_ms=0, max_steps=-first)
        else:
            solver = GpuBoundSolver(engine, encoding, limits, seed=seed, budget_ms=budget_ms)
        solver.add_cnf(cnf)                                     # solver_runner.rs:12
        result = solver.solve()
        if result != SAT and lp_pending:
            lp_done = True                                      # the GPU found nothing below the current count: can the fractional bound certify it?
            # (asked only "does the bound reach the count at hand?": the simplex stops as soon as it does)
            lower = max(lower, engine.lower_bound_lp(g, encoding.defs, target=best.platform_count())["bound"])
            if limits.card_limits.get(one) is not None and limits.card_limits[one] < lower:
                steps.append(dict(bound=limits.card_limits[one], result=UNSAT, source="lower bound"))
                proved = True
                break
            if budget_ms is None and first < give_up:           # not refuted: the whole budget, other seeds
                solver = GpuBoundSolver(engine, encoding, limits, seed=seed ^ 0x9E3779B97F4A7C15, budget_ms=0, max_steps=-give_up)
                solver.add_cnf(cnf)
                result = solver.solve()
        if result == SAT:
            give_up = max(1024, 32 * int(engine.stats()["last_solve_steps"]))
        source = "gpu"
        assignment = solver.full_solution() if result == SAT else None
        if result != SAT and exact_solver is not None:          # the GPU found nothing in budget: ask the prover
            result, assignment = exact_solver(cnf)
            source = "exact"
        bound = limits.card_limits.get(one)
        if result != SAT:                                       # main.rs:331-338
            steps.append(dict(bound=bound, result=result, source=source))
            proved = result == UNSAT and best is not None
            break
        layout = PlatformLayout.from_assignment(assignment, encoding)   # main.rs:328-329
        count = layout.platform_count()
        valid = layout.validate(project.world, engine).is_valid()       # main.rs:353 (warn only)
        steps.append(dict(bound=bound, result=SAT, count=count, valid=valid, source=source))
        if on_solution:
            on_solution(layout)
        best = layout
        if count == 0:                                          # main.rs:341-344
            break
        limits.card_limits[one] = count - 1                     # main.rs:346
    return dict(best=best, proved_optimal=proved, steps=steps, lower_bound=lower)


def weight_loop(project: Project, encoding: Encoding, weights: dict, engine: Engine, exact_solver=None, seed=0, max_steps=4096, use_lower_bound=True):
    """The GUI's loop (crates/gui/src/app.rs:212-249): solve, run_trivial_optimization, weight = total_weight(layout),
    weight_limit = weight - 1, again — until the solver says UNSAT.  The GPU answers the SAT iterations (weighted placement
    search, witness verified against the CNF incl. the PB constraint); the certified fractional bound on the total weight
    (tss_lower_bound_lp with the same weights) ends the loop when the weight meets it; `exact_solver` gets what is left.

    Returns dict(best=PlatformLayout|None, best_weight=int|None, proved_optimal=bool, steps=[...], lower_bound=int|None)."""
    limits = PlatformLimits({}, dict(weights), None)
    steps, best, best_weight, proved = [], None, None, False
    g = encoding._grid
    engine.clear_interrupt()
    lower = None
    if use_lower_bound and g.width <= 32 and g.height <= 32:
        try:
            lower = engine.lower_bound_lp(g, encoding.defs, weights=weights)["bound"]
        except TssError as err:
            if err.code != _lib.TSS_E_UNSUPPORTED:
                raise
    while True:
        if lower is not None and best is not None and limits.weight_limit < lower:
            steps.append(dict(weight_limit=limits.weight_limit, result=UNSAT, source="lower bound"))
            proved = True
            break
        cnf = encoding.with_limits(limits)                      # solver_backend.rs:76-78
        solver = GpuBoundSolver(engine, encoding, limits, seed=seed, budget_ms=0, max_steps=max_steps)
        solver.add_cnf(cnf)
        result = solver.solve()
        source = "gpu"
        assignment = solver.full_solution() if result == SAT else None
        if result != SAT and exact_solver is not None:
            result, assignment = exact_solver(cnf)
            source = "exact"
        if result != SAT:
            steps.append(dict(weight_limit=limits.weight_limit, result=result, source=source))
            proved = result == UNSAT and best is not None
            break
        layout = PlatformLayout.from_assignment(assignment, encoding)   # app.rs:156
        layout.run_trivial_optimization(project.world)                  # app.rs:157
        weight = layout.total_weight(weights)                            # app.rs:235
        steps.append(dict(weight_limit=limits.weight_limit, result=SAT, weight=weight, source=source))
        best, best_weight = layout, weight
        if weight <= 0:
            break
        limits.weight_limit = weight - 1                                 # app.rs:240
    return dict(best=best, best_weight=best_weight, proved_optimal=proved, steps=steps, lower_bound=lower)
