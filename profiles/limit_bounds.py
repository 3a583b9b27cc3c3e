"""The REPL's `solve -l k:v` loops with and without --limit-bounds (the class-aware LP, tss_lower_bound_lp_limits).

For every row: the loop's wall time (the driver's `ms`: encode, bounds, every iteration), its exact-solver calls and verdict,
once without and once with --limit-bounds, and the pivots and device time of the LP each side asks (the plain LP of the whole
set, the class-aware LP run to optimality).  The exact solver is tests/exact_dimacs.py (the oracle's CDCL).

    python profiles/limit_bounds.py [--out FILE.jsonl]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import timberborn_support_solver_b200 as T  # noqa: E402
from conftest import golden, rows_to_grid, synth_terrain  # noqa: E402

FIX = {k: rows_to_grid(v["grid"]) for k, v in golden("fixtures").items()}
ROWS = [("ex2", FIX["ex2"], "5:2"), ("ex2", FIX["ex2"], "5:1,1x6:2"), ("ex2", FIX["ex2"], "3:1"), ("ex2", FIX["ex2"], "1x2:2"),
        ("synth18x16", synth_terrain(18, 16, seed=7, t=3), "5:1,3:2"), ("synth32", synth_terrain(32, 32, seed=1, t=0), "3:4"),
        ("ex1", FIX["ex1"], "5:0,3:0")]


def parse_limits(arg):
    out = {}
    for item in arg.split(","):
        k, v = item.split(":")
        a, b = (k.split("x") + [k])[:2] if "x" in k else (k, k)
        out[T.PlatformDef(min(int(a), int(b)), max(int(a), int(b)))] = int(v)
    return out


def repl(grid, arg, extra, tmp):
    proj = os.path.join(tmp, "project.toml")
    with open(proj, "w") as f:
        f.write(T.WorldGrid(grid).to_toml())
    exe = os.path.join(ROOT, "timberborn_support_solver_b200", "tss_repl")
    exact = f"{sys.executable} {os.path.join(ROOT, 'tests', 'exact_dimacs.py')}"
    t = time.perf_counter()
    out = subprocess.run([exe, proj, "--exact", exact, "-l", arg, "--seed", "3", "--quiet", *extra], capture_output=True, text=True, timeout=3600)
    wall = (time.perf_counter() - t) * 1e3
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("# best=")][-1]
    f = dict(kv.split("=", 1) for kv in re.sub(r'verdict="[^"]*" ', "", line[2:]).split(" ") if "=" in kv)
    verdict = re.search(r'verdict="([^"]*)"', line).group(1)
    return dict(best=int(f["best"]), lower_bound=int(f["lower_bound"]), exact_solves=int(f["exact_solves"]), gpu_solves=int(f["gpu_solves"]),
                loop_ms=float(f["ms"]), process_ms=round(wall, 1), verdict=verdict)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    eng = T.Engine(0)
    dev = eng.device_info()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines = [dict(gpu=smi, **dev)]
    with tempfile.TemporaryDirectory() as tmp:
        for name, grid, arg in ROWS:
            g = T.WorldGrid(grid)
            lp = {}
            for side, lim in (("plain", None), ("limits", parse_limits(arg))):
                eng.lower_bound_lp(g, T.PLATFORMS_DEFAULT, limits=lim)          # warm: scratch slots, modules
                t = time.perf_counter()
                r = eng.lower_bound_lp(g, T.PLATFORMS_DEFAULT, limits=lim)
                lp[side] = dict(bound=r["bound"], pivots=r["pivots"], optimal=r["optimal"], constraints=r["constraints"],
                                wall_ms=round((time.perf_counter() - t) * 1e3, 3), device_ms=round(eng.stats()["device_ms"], 3))
            # (the loops on 32x32 are left out: without the class bound their last UNSAT goes to the exact solver, which does not
            # finish there)
            loops = {} if grid.shape[0] > 24 else {side: repl(grid, arg, extra, tmp) for side, extra in (("off", ()), ("limit_bounds", ("--limit-bounds",)))}
            row = dict(terrain=name, limits=arg, lp=lp, loop=loops)
            print(json.dumps(row), flush=True)
            lines.append(row)
    eng.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
