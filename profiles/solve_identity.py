"""A fixed, seeded sequence of one-shot calls on ONE engine, so that its cached workspaces are created, reused, adopted and
dropped in a known order, with one JSON record per call: the result code, the sorted layout, the engine's last error text and
`stats()` without `device_ms` (the one counter that is a time).  Two builds of libtss that must compute the same thing write
byte-identical files.

    python profiles/solve_identity.py OUT.json                        (the library built in this tree)
    TSS_LIB=path/to/other/libtss.so python profiles/solve_identity.py OTHER.json
    cmp OUT.json OTHER.json

The sequence:
  * solve_upper_bound on rect 16x16 and test/ex1-3, unbounded and then with bound = found - 1, with 1x1 and with the default-8
    set (cold calls, then the fused first epochs on the cached workspaces, then a change of platform set); then default-8
    against its first four defs on test/ex2 (the placement workspace adopted for other keys);
  * 1x1 with a step budget (the 1x1 workspace replaced for another chain count, then reused without the fused epoch);
  * a bound no layout meets, with max_steps = -300 (the give-up point), on 1x1 and default-8;
  * solve_with_limits with per-type limits, and with a limit of 0 (the class dropped from the set);
  * a weighted solve_with_limits that fails on a weight of 0 (the cached placement workspace adopted, then destroyed);
    solve_min_weight twice with a tightening weight limit, then a solve_upper_bound with a step budget on the same set (same
    chain count: tss_search_create adopts the weighted workspace);
  * lower_bound and lower_bound_lp (plain and weighted) on rect 16x16 and on a synthetic 48x40 grid;
  * one failing call per platform-set check and per weight range check."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import timberborn_support_solver_b200 as T  # noqa: E402
from conftest import golden, rows_to_grid, synth_terrain  # noqa: E402

P = T.PlatformDef
D8 = list(T.PLATFORMS_DEFAULT)
ONE = D8[:1]


def layout_rows(layout):
    return sorted((p.x, p.y, p.definition.width, p.definition.height, int(p.rotated)) for p in layout.platforms().values()) if layout else None


def main():
    out = sys.argv[1]
    fx = {k: rows_to_grid(v["grid"]) for k, v in golden("fixtures").items()}
    grids = {"rect16": np.ones((16, 16), np.uint8), **fx}
    big = synth_terrain(48, 40, seed=3, t=1)
    e = T.Engine(0)
    records = []

    def call(label, fn, *args, **kw):
        rec = {"call": label}
        try:
            r = fn(*args, **kw)
            rec["result"], rec["value"] = r[0] if isinstance(r, tuple) else "ok", r
        except T.TssError as err:
            rec["result"], rec["value"] = err.code, None
        rec["error"] = e.lib.tss_last_error(e._h).decode()
        rec["stats"] = {k: v for k, v in e.stats().items() if k != "device_ms"}
        records.append(rec)
        return rec["value"]

    def solve(label, g, defs, limit=None, **kw):
        def fn():
            res, lay = e.solve_upper_bound(T.WorldGrid(g), defs, card_limit=limit, **kw)
            return res, layout_rows(lay)
        v = call(label, fn)
        return None if v is None or v[1] is None else len(v[1])

    for defs_name, defs in (("1x1", ONE), ("default-8", D8)):
        for name, g in grids.items():
            found = solve(f"solve_upper_bound {name} {defs_name} unbounded", g, defs, seed=7)
            if found:
                solve(f"solve_upper_bound {name} {defs_name} bound {found - 1}", g, defs, found - 1, seed=8)
    solve("solve_upper_bound ex2 default-8[:4] unbounded", grids["ex2"], D8[:4], seed=9)
    solve("solve_upper_bound ex2 default-8 bound 4", grids["ex2"], D8, 4, seed=9)
    for name in ("rect16", "ex2", "rect16"):   # a step budget: other chain counts (the 1x1 workspace replaced, then reused without a fused epoch)
        solve(f"solve_upper_bound {name} 1x1 max_steps 2000", grids[name], ONE, seed=15, max_steps=2000)
    solve("solve_upper_bound rect16 1x1 bound 10 max_steps -300", grids["rect16"], ONE, 10, seed=10, max_steps=-300)
    solve("solve_upper_bound ex2 default-8 bound 1 max_steps -300", grids["ex2"], D8, 1, seed=10, max_steps=-300)

    def with_limits(label, g, defs, limits, wts=None):
        def fn():
            res, lay, obj = e.solve_with_limits(T.WorldGrid(g), defs, T.PlatformLimits(limits, wts or {}), seed=11)
            return res, layout_rows(lay), obj
        call(label, fn)

    with_limits("solve_with_limits ex2 default-8 5x5<=1 3x3<=1", grids["ex2"], D8, {P(5, 5): 1, P(3, 3): 1})
    with_limits("solve_with_limits ex2 default-8 5x5<=0", grids["ex2"], D8, {P(5, 5): 0})
    with_limits("solve_with_limits rect16 default-8 1x1<=20 1x6<=2", grids["rect16"], D8, {P(1, 1): 20, P(1, 6): 2})

    weights = {P(1, 1): 1, P(1, 2): 2, P(1, 3): 3, P(1, 4): 3, P(1, 5): 4, P(1, 6): 4, P(3, 3): 6, P(5, 5): 9}

    def min_weight(label, g, limit, wts=weights):
        def fn():
            res, lay, wt = e.solve_min_weight(T.WorldGrid(g), D8, wts, weight_limit=limit, seed=12)
            return res, layout_rows(lay), wt
        v = call(label, fn)
        return None if v is None else v[2]

    # a weight of 0 fails after tss_search_create adopted the cached placement workspace: it is destroyed, the slot is free
    with_limits("solve_with_limits ex2 default-8 a weight of 0", grids["ex2"], D8, {}, {P(1, 1): 0})
    wt = min_weight("solve_min_weight ex2 unbounded", grids["ex2"], None)
    if wt:
        min_weight(f"solve_min_weight ex2 limit {wt - 1}", grids["ex2"], wt - 1)
    solve("solve_upper_bound ex2 default-8 max_steps 2000 (adopts the weighted workspace)", grids["ex2"], D8, seed=13, max_steps=2000)
    solve("solve_upper_bound ex2 default-8 unbounded (after the adoption)", grids["ex2"], D8, seed=14)

    def lower_bound(label, g, defs):
        call(label, lambda: e.lower_bound(T.WorldGrid(g), defs, seed=5))

    def lower_bound_lp(label, g, defs, wts=None):
        def fn():
            r = e.lower_bound_lp(T.WorldGrid(g), defs, weights=wts)
            r["weights"] = hashlib.sha256(np.ascontiguousarray(r["weights"]).tobytes()).hexdigest()
            return r
        call(label, fn)

    lower_bound("lower_bound rect16 default-8", grids["rect16"], D8)
    lower_bound("lower_bound 48x40 1x1", big, ONE)
    lower_bound_lp("lower_bound_lp rect16 1x1", grids["rect16"], ONE)
    lower_bound_lp("lower_bound_lp ex2 default-8 weighted", grids["ex2"], D8, weights)
    lower_bound_lp("lower_bound_lp 48x40 default-8 weighted", big, D8, weights)
    lower_bound_lp("lower_bound_lp 48x40 1x1", big, ONE)

    no_1x1, empty = [P(1, 2), P(3, 3)], [P(1, 1), P(0, 2)]
    solve("solve_upper_bound without 1x1", grids["ex1"], no_1x1)
    solve("solve_upper_bound empty def", grids["ex1"], empty)
    call("search without 1x1", lambda: e.search(T.WorldGrid(grids["ex1"]), no_1x1) and None)
    lower_bound("lower_bound without 1x1", grids["ex1"], no_1x1)
    lower_bound("lower_bound empty def", grids["ex1"], empty)
    lower_bound_lp("lower_bound_lp without 1x1", grids["ex1"], no_1x1)
    lower_bound_lp("lower_bound_lp empty def", grids["ex1"], empty)
    min_weight("solve_min_weight a weight of 0", grids["ex1"], None, {P(1, 1): 0})
    lower_bound_lp("lower_bound_lp a weight over 4096", grids["ex1"], D8, {P(1, 1): 5000})
    e.close()
    with open(out, "w") as f:
        for rec in records:
            f.write(json.dumps(rec, sort_keys=True) + "\n")
    print(f"{len(records)} calls -> {out}")


if __name__ == "__main__":
    main()
