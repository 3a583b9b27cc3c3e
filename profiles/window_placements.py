"""The window-decomposed placement search (TSS_KERNEL_WINDOW_PLACEMENTS) against AUTO (the 1x1 window decomposition plus the
host post-pass: supports merged under footprints / greedy placement cover, whichever has fewer platforms) on grids larger
than 32x32, at equal phases: 16 phases of 2 000 steps, 3 seeds, default chains per window.  Per run: the final objective
(platform count, or total weight with the GUI weights) and the device time per phase (the engine's CUDA events around each
tss_search_run, after a warm-up run of both searches).  AUTO cannot search the weight objective on these grids: its row
reports the total weight of its platform-count layout.

python profiles/window_placements.py [--out FILE]"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import timberborn_support_solver_b200 as T  # noqa: E402
from conftest import synth_terrain  # noqa: E402

PHASES, STEPS, SEEDS = 16, 2000, (1, 2, 3)
GUI_WEIGHTS = {T.PlatformDef(1, 1): 3, T.PlatformDef(1, 3): 2, T.PlatformDef(3, 3): 4, T.PlatformDef(5, 5): 7}
TERRAINS = [  # (name, w, h, density, seed, t, weights): the three terrains of blocks_experiment.py (256x256 p = 0.7 is SURVEY.md C4)
    ("dense 96x72", 96, 72, 0.85, 4, 1, None),
    ("128x128 p=0.7", 128, 128, 0.7, 1, 0, None),
    ("C4 256x256 p=0.7", 256, 256, 0.7, 1, 0, None),
    ("dense 96x72, GUI weights", 96, 72, 0.85, 4, 1, GUI_WEIGHTS),
]


def total_weight(layout, weights):
    canon = lambda w, h: (min(w, h), max(w, h))
    tot = 0
    for p in layout.platforms().values():
        cw, ch = canon(p.definition.width, p.definition.height)
        tot += sum(v for d, v in weights.items() if canon(d.width, d.height)[0] <= cw and canon(d.width, d.height)[1] <= ch)
    return tot


def run(eng, grid, kernel, seed, weights, phases=PHASES):
    s = eng.search(grid, T.PLATFORMS_DEFAULT, seed=seed, kernel=kernel)
    if weights and kernel == T.KERNEL_WINDOW_PLACEMENTS:
        s.set_weights(weights)
    ms = []
    for _ in range(phases):
        s.run(STEPS, 0)
        s.best_count()                                   # synchronises; device_ms = the phase's CUDA events
        ms.append(eng.stats()["device_ms"])
    t0 = time.perf_counter()
    lay = s.best_layout()
    host_ms = (time.perf_counter() - t0) * 1e3
    s.close()
    obj = total_weight(lay, weights) if weights else lay.platform_count()
    return obj, float(np.mean(ms)), host_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(msg):
        print(msg, flush=True)
        lines.append(msg)
    eng = T.Engine(0)
    info = eng.device_info()
    say(f"# python profiles/window_placements.py: {info.get('name', '?')}; {PHASES} phases x {STEPS} steps, seeds {SEEDS}, default chains per window")
    for name, w, h, dens, tseed, t, weights in TERRAINS:
        grid = T.WorldGrid(synth_terrain(w, h, seed=tseed, t=t, density_q24=int(dens * (1 << 24))))
        for kernel in (T.KERNEL_AUTO, T.KERNEL_WINDOW_PLACEMENTS):   # warm-up: module loads, allocations
            run(eng, grid, kernel, 0, weights, phases=1)
        for kernel, label in ((T.KERNEL_AUTO, "AUTO (1x1 LNS + post-pass)"), (T.KERNEL_WINDOW_PLACEMENTS, "window placements (kernel 5)")):
            res = [run(eng, grid, kernel, seed, weights) for seed in SEEDS]
            objs = [r[0] for r in res]
            say(f"{name:26s} {label:30s} objective {objs} (mean {np.mean(objs):.1f}); device {np.mean([r[1] for r in res]):.2f} ms per phase; "
                f"best_layout host {np.mean([r[2] for r in res]):.1f} ms")
    eng.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
