"""TEST INFRASTRUCTURE ONLY: scalar replay of the window-decomposed placement search with per-type platform limits
(tss_search_create_with_limits: csrc/lns_placements.cu driving sls_multi_kernel<false, true, true>) for the tests.  The global
part — the start layout trimmed to the limits, the per-window class budgets, the movable / frozen split, cut, winner and
write-back — is restated here in numpy; the windows' chains run through tests/window_limits_model.cpp (the WINDOW step-rule
replay of tests/window_model.cpp with the class counters), compiled on first use into a per-user temporary directory (the
repository tree is never written)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from window_model import _grid, _i32, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "window_limits_model.cpp")
_lib = None

CORE_LO, CORE_HI = 3, 29
OFF = [(0, 0), (-16, -16), (0, -16), (-16, 0)]


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for src in (_SRC, os.path.join(_HERE, "window_model.cpp")):
            with open(src, "rb") as f:
                h.update(f.read())
        out_dir = os.path.join(tempfile.gettempdir(), f"tss_window_limits_model_{os.getuid()}")
        so = os.path.join(out_dir, f"window_limits_model_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-Wall", "-shared", "-o", tmp, _SRC])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def reach(C_, x, y, pw, ph):
    """validate()'s reach of one footprint: three ceiling-masked 4-neighbour dilations from the ceiling under it -> bool[h, w]"""
    h, w = C_.shape
    r = np.zeros((h, w), bool)
    r[y:y + ph, x:x + pw] = C_[y:y + ph, x:x + pw] != 0
    for _ in range(3):
        nb = r.copy()
        nb[:, 1:] |= r[:, :-1]; nb[:, :-1] |= r[:, 1:]; nb[1:, :] |= r[:-1, :]; nb[:-1, :] |= r[1:, :]
        r = nb & (C_ != 0)
    return r


def limit_start(grid, key_dims, start, key_mask, class_limit):
    """The start layout under per-type limits: the platforms of `start` in row-major anchor order, each kept only while every
    class it belongs to has room, then a 1x1 on every ceiling tile (row-major) still unsupported.  start: [(x, y, key)]
    -> sorted [(x, y, key)]"""
    C_ = _grid(grid)
    h, w = C_.shape
    one = list(map(tuple, np.asarray(key_dims).reshape(-1, 2).tolist())).index((1, 1))
    n = [0] * len(class_limit)
    sup = np.zeros((h, w), bool)
    kept = []
    for x, y, k in sorted(start, key=lambda p: (p[1], p[0])):
        m = int(key_mask[k])
        if any((m >> j) & 1 and n[j] >= class_limit[j] for j in range(len(class_limit))):
            continue
        for j in range(len(class_limit)):
            n[j] += (m >> j) & 1
        kept.append((x, y, k))
        sup |= reach(C_, x, y, *key_dims[k])
    for y in range(h):
        for x in range(w):
            if C_[y, x] and not sup[y, x]:
                kept.append((x, y, one))
                sup |= reach(C_, x, y, 1, 1)
    return sorted(kept)


def class_counts(layout, key_mask, n_classes):
    return [sum((int(key_mask[k]) >> j) & 1 for _, _, k in layout) for j in range(n_classes)]


def window_budgets(n_windows, phase, slack, movable):
    """b_{w,j} = m_{w,j} + floor(s_j / N) + [((w - p) mod N) < (s_j mod N)]; movable[w][j] = m_{w,j} -> int[N][n_classes]"""
    N = n_windows
    return np.array([[movable[w][j] + s // N + (1 if (w - phase) % N < s % N else 0) for j, s in enumerate(slack)] for w in range(N)], np.int64)


def lns_placements_limits_model(grid, key_dims, costs, start, seeds, phases, phase_steps, key_mask, class_limit, seed=0, chain_offset=0,
                                noise_pct=20):
    """lns_placements_model (tests/window_model.py) with per-type limits: key_mask[k] = classes of key k (bit j = class j),
    class_limit[j] = L_j; `start` keeps every limit (limit_start).  At the start of phase p, n_j = the layout's platforms in class
    j, m_{w,j} = window w's movable platforms in class j, s_j = L_j - n_j, and window w's chains run with class budgets b_{w,j}
    (window_budgets).
    -> dict(layouts, objectives, budgets=[int[N][n_classes] per phase], frozen=[[n_j - sum_w m_{w,j}] per phase],
            counts=[[n_j after the phase] per phase], binding=[a class of some chain was full, per phase], scored_total, steps_total,
            flips_total)"""
    assert phase_steps <= 32768
    C_ = _grid(grid).astype(np.uint8)
    h, w = C_.shape
    kd = np.ascontiguousarray(key_dims, np.int32).reshape(-1, 2)
    cs = np.ascontiguousarray(costs, np.int32)
    mk = np.ascontiguousarray(key_mask, np.int32)
    nc = len(class_limit)
    anchors = {(int(x), int(y)): int(k) for x, y, k in start}
    layouts, objectives, budgets, frozen, counts, binding = [], [], [], [], [], []
    totals = np.zeros(3, np.uint64)
    L = lib()
    for phase in range(phases):
        ox, oy = OFF[phase & 3]
        nwx, nwy = (w - ox + 31) // 32, (h - oy + 31) // 32
        N = nwx * nwy
        Ff = np.zeros((h, w), np.uint8)
        movable = {}
        for (x, y), k in anchors.items():
            pw, ph = kd[k]
            lx, ly = (x - ox) % 32, (y - oy) % 32
            if CORE_LO <= lx and lx + pw <= CORE_HI and CORE_LO <= ly and ly + ph <= CORE_HI:
                movable.setdefault(((y - oy) // 32) * nwx + (x - ox) // 32, []).append((y, x, k))
            else:
                Ff[y:y + ph, x:x + pw] = 1
        n_now = class_counts([(x, y, k) for (x, y), k in anchors.items()], mk, nc)
        m = [[sum((int(mk[k]) >> j) & 1 for _, _, k in movable.get(win, [])) for j in range(nc)] for win in range(N)]
        slack = [class_limit[j] - n_now[j] for j in range(nc)]
        assert min(slack, default=0) >= 0
        b = window_budgets(N, phase, slack, m)
        budgets.append(b)
        binding.append(False)
        frozen.append([n_now[j] - sum(m[win][j] for win in range(N)) for j in range(nc)])
        cov = Ff & C_
        for _ in range(3):
            nb = cov.copy()
            nb[:, 1:] |= cov[:, :-1]; nb[:, :-1] |= cov[:, 1:]; nb[1:, :] |= cov[:-1, :]; nb[:-1, :] |= cov[1:, :]
            cov = nb & C_
        moved = {(x, y) for ms in movable.values() for y, x, _ in ms}
        new = {p: k for p, k in anchors.items() if p not in moved}
        for win in range(N):
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
            bw = _i32(b[win])
            best_items = np.zeros((seeds, 1024), np.uint16)
            best_k, best = np.zeros(seeds, np.int32), np.zeros(seeds, np.int32)
            ncls, bind = np.zeros((seeds, 16), np.int32), np.zeros(seeds, np.int32)
            rc = L.tsso_slsm_window_limits_model(_p(c, C.c_uint8), _p(need, C.c_uint8), _p(occ, C.c_uint8), _p(box), _p(kd), _p(cs), len(cs), seeds,
                                                 C.c_uint32(chain_offset + win * seeds), C.c_uint64(seed), noise_pct, C.c_longlong(phase_steps),
                                                 _p(codes, C.c_uint16), len(items), best0, C.c_uint32(((phase + 1) << 20) & 0xffffffff), _p(mk), _p(bw), nc,
                                                 _p(best_items, C.c_uint16), _p(best_k), _p(best), _p(ncls), _p(bind), _p(totals, C.c_uint64))
            assert rc == 0
            assert (ncls[:, :nc] <= b[win][None, :]).all()   # every chain's best keeps its window's budgets
            binding[-1] = binding[-1] or bool(bind.any())
            winner = int(np.argmin(best))
            for code in best_items[winner, :best_k[winner]]:
                code = int(code)
                new[(gx0 + (code & 31), gy0 + ((code >> 5) & 31))] = code >> 10
        anchors = new
        lay = sorted((x, y, k) for (x, y), k in anchors.items())
        layouts.append(lay)
        objectives.append(int(sum(int(cs[k]) for k in anchors.values())))
        counts.append(class_counts(lay, mk, nc))
    return dict(layouts=layouts, objectives=objectives, budgets=budgets, frozen=frozen, counts=counts, binding=binding, scored_total=int(totals[0]),
                steps_total=int(totals[1]), flips_total=int(totals[2]))
