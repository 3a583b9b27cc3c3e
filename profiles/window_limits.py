"""Per-type limits in the window placement search (tss_search_create_with_limits) on grids larger than 32x32, in the setting of
profiles/window_placements.py: 16 phases of 2 000 steps, seeds 1-3, default chains per window, the default-8 set, on SURVEY.md C4
(256x256, p = 0.7) and the dense 96x72 terrain.

  1. device time per phase (the engine's CUDA events around each tss_search_run) without limits and with `-l 5:2`, the two
     searches alternated seed by seed in one process after a warm-up run of each;
  2. the count reached under `-l 5:k` and `-l 1x2:k` (the class of every key but 1x1) for a few k;
  3. the wall time of `tss_repl --window-limits -l 5:2` on a 48x48 project until the GPU gives up (no exact solver).

The card's name and power limit are read in the same call (nvidia-smi, read-only query).

python profiles/window_limits.py [--out FILE]"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import timberborn_support_solver_b200 as T  # noqa: E402
from conftest import synth_terrain  # noqa: E402

P = T.PlatformDef
PHASES, STEPS, SEEDS = 16, 2000, (1, 2, 3)
TERRAINS = [("C4 256x256 p=0.7", 256, 256, 0.7, 1, 0), ("dense 96x72", 96, 72, 0.85, 4, 1)]
SWEEP = [("5:1", {P(5, 5): 1}), ("5:4", {P(5, 5): 4}), ("5:16", {P(5, 5): 16}), ("1x2:25", {P(1, 2): 25}), ("1x2:100", {P(1, 2): 100}),
         ("1x2:400", {P(1, 2): 400})]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "not read"


def run(eng, grid, seed, limits, phases=PHASES):
    """-> (count, mean device ms per phase)"""
    kw = dict(limits=limits) if limits else dict(kernel=T.KERNEL_WINDOW_PLACEMENTS)
    s = eng.search(grid, T.PLATFORMS_DEFAULT, seed=seed, **kw)
    ms = []
    for _ in range(phases):
        s.run(STEPS, -1)
        s.best_count()                                   # synchronises; device_ms = this phase's events
        ms.append(eng.stats()["device_ms"])
    c = s.best_layout().platform_count()
    s.close()
    return c, float(np.mean(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(msg):
        print(msg, flush=True)
        lines.append(msg)
    eng = T.Engine(0)
    say(f"# python profiles/window_limits.py: {PHASES} phases x {STEPS} steps, seeds {SEEDS}, default chains per window, default-8 set")
    say(f"# card: {card()} (name, power limit, max SM clock, read in the same call)")
    for name, w, h, dens, tseed, t in TERRAINS:
        grid = T.WorldGrid(synth_terrain(w, h, seed=tseed, t=t, density_q24=int(dens * (1 << 24))))
        run(eng, grid, 0, None, phases=1)                   # warm-up: module loads, allocations
        run(eng, grid, 0, {P(5, 5): 2}, phases=1)
        res = {"none": [], "5:2": []}
        for seed in SEEDS:                                  # alternated seed by seed
            res["none"].append(run(eng, grid, seed, None))
            res["5:2"].append(run(eng, grid, seed, {P(5, 5): 2}))
        for label, r in res.items():
            say(f"{name:18s} limits {label:8s} count {[c for c, _ in r]}; device {np.mean([m for _, m in r]):.2f} ms per phase "
                f"({', '.join(f'{m:.2f}' for _, m in r)})")
        for label, lim in SWEEP:
            r = [run(eng, grid, seed, lim) for seed in SEEDS]
            say(f"{name:18s} limits {label:8s} count {[c for c, _ in r]} (mean {np.mean([c for c, _ in r]):.1f}); device {np.mean([m for _, m in r]):.2f} ms per phase")
    eng.close()
    with tempfile.TemporaryDirectory() as d:
        proj = os.path.join(d, "project.toml")
        with open(proj, "w") as f:
            f.write(T.WorldGrid(synth_terrain(48, 48, seed=2, t=1)).to_toml())
        exe = os.path.join(os.path.dirname(T.__file__), "tss_repl")
        t0 = time.perf_counter()
        out = subprocess.run([exe, proj, "--window-limits", "-l", "5:2", "--seed", "3", "--quiet"], capture_output=True, text=True, timeout=600)
        wall = (time.perf_counter() - t0) * 1e3
        summary = [ln for ln in out.stdout.splitlines() if ln.startswith("# best=")]
        say(f"tss_repl --window-limits -l 5:2, 48x48 (synth seed 2, t 1): wall {wall:.0f} ms (process, engine start-up included); "
            f"{summary[-1] if summary else out.stderr.strip()}")
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
