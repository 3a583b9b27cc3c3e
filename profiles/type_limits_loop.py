"""The REPL's `solve -l k:v` loop with per-type platform limits: the C++ driver (timberborn_support_solver_b200/tss_repl) to
the PROVEN optimum over the C ABI, `--repeat 11` (cold first run, warm median of the rest, the oracle's CDCL as `--exact`),
against the oracle's CPU-only loop under the same limits (CDCL on every iteration, crates/repl/src/main.rs:280-366).
Records wall times, GPU / exact-solver calls, the card and its power limit.

    python profiles/type_limits_loop.py > profiles/r11_type_limits_loop.json
"""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle.oracle as O                      # noqa: E402
import timberborn_support_solver_b200 as T   # noqa: E402
from conftest import golden, rows_to_grid, synth_terrain   # noqa: E402

CASES = [("ex1", "3:1,1x4:2", {(3, 3): 1, (1, 4): 2}), ("ex2", "5:2", {(5, 5): 2}), ("ex2", "5:1,1x6:2", {(5, 5): 1, (1, 6): 2}),
         ("ex3", "3:2,1x2:3", {(3, 3): 2, (1, 2): 3}), ("random", "5:1,3:2", {(5, 5): 1, (3, 3): 2})]


def cpu_loop(grid, card):
    """-> (optimum, CDCL calls, wall ms)"""
    t0 = time.perf_counter()
    enc = O.Encoding(O.PLATFORMS_DEFAULT, grid)
    best, calls, limits = None, 0, dict(card)
    while True:
        r, a, _ = enc.with_limits(card_limits=limits).solve()
        calls += 1
        if r != 10:
            return best, calls, (time.perf_counter() - t0) * 1e3
        best = len(enc.layout_from_assignment(a))
        limits[(1, 1)] = best - 1


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = {"gpu": smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "unavailable"}
    exe = os.path.join(os.path.dirname(T.__file__), "tss_repl")
    exact = f"{sys.executable} {os.path.join(ROOT, 'tests', 'exact_dimacs.py')}"
    grids = {k: rows_to_grid(v["grid"]) for k, v in golden("fixtures").items()}
    grids["random"] = synth_terrain(18, 16, seed=7, t=3)
    with tempfile.TemporaryDirectory() as tmp:
        for name, arg, card in CASES:
            path = os.path.join(tmp, name + ".toml")
            with open(path, "w") as f:
                f.write(T.WorldGrid(grids[name]).to_toml())
            r = subprocess.run([exe, path, "-l", arg, "--exact", exact, "--seed", "3", "--quiet", "--repeat", "11"], capture_output=True, text=True, timeout=1200)
            lines = [ln for ln in r.stdout.splitlines() if ln.startswith("# ")]
            opt, calls, ms = cpu_loop(grids[name], card)
            out[f"{name} -l {arg}"] = {"gpu_loop": lines[0] if r.returncode == 0 and lines else r.stderr[-300:],
                                        "cpu_loop": {"best": opt, "cdcl_calls": calls, "ms": round(ms, 1)}}
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
