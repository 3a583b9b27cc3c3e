"""TEST INFRASTRUCTURE ONLY: scalar replay of the window-decomposed placement search (TSS_KERNEL_WINDOW_PLACEMENTS,
timberborn_support_solver_b200/csrc/lns_placements.cu) for the tests.  The global part (movable / frozen split, footprint
stamp, frozen cover, window cut, row-major item order, winner, write-back) is restated here in numpy; the windows' chains run
through the scalar step-rule replay in tests/window_model.cpp, compiled on first use into a per-user temporary directory
(the repository tree is never written)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "window_model.cpp")
_lib = None


def lib():
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"tss_window_model_{os.getuid()}")
        so = os.path.join(out_dir, f"window_model_{tag}.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-Wall", "-shared", "-o", tmp, _SRC])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _grid(grid):
    g = np.ascontiguousarray(grid, dtype=np.uint8)
    assert g.ndim == 2
    return g


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a, t=C.c_int):
    return a.ctypes.data_as(C.POINTER(t))


def lns_placements_model(grid, key_dims, costs, start, seeds, phases, phase_steps, seed=0, chain_offset=0, noise_pct=20):
    """Scalar replay of the window-decomposed placement search for grids larger than 32x32
    (timberborn_support_solver_b200/csrc/lns_placements.cu).  key_dims: [(w, h)] effective dims per key in the engine's key
    order, costs: objective cost per key, start: the start layout as [(x, y, key)] (complete, footprints in bounds and
    disjoint).  Phase p tiles the grid with 32x32 windows at offset OFF[p & 3]; a platform is movable iff its footprint lies
    in its window's [3, 29)^2, every other platform is frozen; in every window `seeds` chains of the WINDOW-mode step rule
    (tests/window_model.cpp) start from the window's movable platforms in row-major anchor order, and the chain with the
    lowest best (lowest chain on ties) replaces them.  phase_steps <= 32768 (one epoch per phase).
    -> dict(layouts=[sorted [(x, y, key)] after every phase], objectives=[...], scored_total, steps_total, flips_total)"""
    assert phase_steps <= 32768
    C_ = _grid(grid).astype(np.uint8)
    h, w = C_.shape
    kd = np.ascontiguousarray(key_dims, np.int32).reshape(-1, 2)
    cs = np.ascontiguousarray(costs, np.int32)
    CORE_LO, CORE_HI = 3, 29
    OFF = [(0, 0), (-16, -16), (0, -16), (-16, 0)]
    anchors = {(int(x), int(y)): int(k) for x, y, k in start}
    layouts, objectives = [], []
    totals = np.zeros(3, np.uint64)
    L = lib()
    for phase in range(phases):
        ox, oy = OFF[phase & 3]
        nwx, nwy = (w - ox + 31) // 32, (h - oy + 31) // 32
        Ff = np.zeros((h, w), np.uint8)
        movable = {}                                         # window -> [(y, x, key)]
        for (x, y), k in anchors.items():
            pw, ph = kd[k]
            lx, ly = (x - ox) % 32, (y - oy) % 32
            if CORE_LO <= lx and lx + pw <= CORE_HI and CORE_LO <= ly and ly + ph <= CORE_HI:
                movable.setdefault(((y - oy) // 32) * nwx + (x - ox) // 32, []).append((y, x, k))
            else:
                Ff[y:y + ph, x:x + pw] = 1
        cov = Ff & C_                                        # exact geodesic cover of the frozen platforms
        for _ in range(3):
            nb = cov.copy()
            nb[:, 1:] |= cov[:, :-1]; nb[:, :-1] |= cov[:, 1:]; nb[1:, :] |= cov[:-1, :]; nb[:-1, :] |= cov[1:, :]
            cov = nb & C_
        moved = {(x, y) for ms in movable.values() for y, x, _ in ms}
        new = {p: k for p, k in anchors.items() if p not in moved}
        for win in range(nwx * nwy):
            gx0, gy0 = ox + 32 * (win % nwx), oy + 32 * (win // nwx)

            def cut(X):
                W_ = np.zeros((32, 32), np.uint8)
                x0, x1, y0, y1 = max(gx0, 0), min(gx0 + 32, w), max(gy0, 0), min(gy0 + 32, h)
                if x1 > x0 and y1 > y0:
                    W_[y0 - gy0:y1 - gy0, x0 - gx0:x1 - gx0] = X[y0:y1, x0:x1]
                return np.ascontiguousarray(W_)
            c, occ = cut(C_), cut(Ff)
            need = np.ascontiguousarray(c & (1 - cut(cov)))
            box = _i32([max(CORE_LO, -gx0), max(CORE_LO, -gy0), min(CORE_HI, w - gx0), min(CORE_HI, h - gy0)])
            items = sorted(movable.get(win, []))
            codes = np.ascontiguousarray([(k << 10) | ((y - gy0) << 5) | (x - gx0) for y, x, k in items] or [0], np.uint16)
            best0 = int(sum(int(cs[k]) for _, _, k in items))
            best_items = np.zeros((seeds, 1024), np.uint16)
            best_k, best = np.zeros(seeds, np.int32), np.zeros(seeds, np.int32)
            rc = L.tsso_slsm_window_model(_p(c, C.c_uint8), _p(need, C.c_uint8), _p(occ, C.c_uint8), _p(box), _p(kd), _p(cs), len(cs), seeds,
                                          C.c_uint32(chain_offset + win * seeds), C.c_uint64(seed), noise_pct, C.c_longlong(phase_steps),
                                          _p(codes, C.c_uint16), len(items), best0, C.c_uint32(((phase + 1) << 20) & 0xffffffff),
                                          _p(best_items, C.c_uint16), _p(best_k), _p(best), _p(totals, C.c_uint64))
            assert rc == 0
            winner = int(np.argmin(best))                    # lowest chain on ties
            for code in best_items[winner, :best_k[winner]]:
                code = int(code)
                new[(gx0 + (code & 31), gy0 + ((code >> 5) & 31))] = code >> 10
        anchors = new
        layouts.append(sorted((x, y, k) for (x, y), k in anchors.items()))
        objectives.append(int(sum(int(cs[k]) for k in anchors.values())))
    return dict(layouts=layouts, objectives=objectives, scored_total=int(totals[0]), steps_total=int(totals[1]),
                flips_total=int(totals[2]))
