"""The fractional lower bound on grids larger than 32x32 (tss_lower_bound_lp, csrc/lp_big.cu) on the large instances, beside what
the searches reach there.  Per instance: the device time of the call (the engine's CUDA events around reach windows, iterations
and certificate, after a warm-up call), the iterations, the certified bound, the time per iteration (difference against a
50-iteration call), the packing bound where one exists (1x1 supports), and the search result at the settings of
window_placements.py (window placement search: 16 phases x 2 000 steps, seeds 1-3) or, for 1x1 supports, of the C4 row of
DESIGN §0 (the 1x1 window search: 16 phases x 4 000 steps, seeds 1-3).  The card's name and power limit are read in the same run.

python profiles/lp_large.py [--out FILE]"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import timberborn_support_solver_b200 as T  # noqa: E402
from conftest import synth_terrain  # noqa: E402

GUI_WEIGHTS = {T.PlatformDef(1, 1): 3, T.PlatformDef(1, 3): 2, T.PlatformDef(3, 3): 4, T.PlatformDef(5, 5): 7}   # window_placements.py's
SEEDS = (1, 2, 3)
INSTANCES = [  # (name, grid, defs, weights)
    ("C4 256x256, 1x1", lambda: synth_terrain(256, 256, seed=1, t=0), T.PLATFORMS_DEFAULT[:1], None),
    ("C4 256x256, default-8", lambda: synth_terrain(256, 256, seed=1, t=0), T.PLATFORMS_DEFAULT, None),
    ("C4 256x256, default-8, GUI weights", lambda: synth_terrain(256, 256, seed=1, t=0), T.PLATFORMS_DEFAULT, GUI_WEIGHTS),
    ("dense 96x72, default-8, GUI weights", lambda: synth_terrain(96, 72, seed=4, t=1, density_q24=int(0.85 * (1 << 24))), T.PLATFORMS_DEFAULT, GUI_WEIGHTS),
]


def total_weight(layout, weights):
    canon = lambda w, h: (min(w, h), max(w, h))
    tot = 0
    for p in layout.platforms().values():
        cw, ch = canon(p.definition.width, p.definition.height)
        tot += sum(v for d, v in weights.items() if canon(d.width, d.height)[0] <= cw and canon(d.width, d.height)[1] <= ch)
    return tot


def search(eng, grid, defs, weights, seed):
    one = len(defs) == 1
    s = eng.search(grid, defs, seed=seed, kernel=T.KERNEL_AUTO if one else T.KERNEL_WINDOW_PLACEMENTS)
    if weights:
        s.set_weights(weights)
    for _ in range(16):
        s.run(4000 if one else 2000, 0)
    lay = s.best_layout()
    s.close()
    return total_weight(lay, weights) if weights else lay.platform_count()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def say(msg):
        print(msg, flush=True)
        lines.append(msg)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    say("# python profiles/lp_large.py: tss_lower_bound_lp on grids larger than 32x32 (first-order method, integer certificate)")
    say(f"# card: {card.splitlines()[0] if card else '?'} (name, power limit, max SM clock, read in the same run)")
    eng = T.Engine(0)
    for name, make, defs, weights in INSTANCES:
        grid = T.WorldGrid(make())
        eng.lower_bound_lp(grid, defs, weights=weights, max_pivots=50)    # warm-up: module load, scratch allocation
        short = eng.lower_bound_lp(grid, defs, weights=weights, max_pivots=50)
        short_ms = eng.stats()["device_ms"]
        r = eng.lower_bound_lp(grid, defs, weights=weights)
        ms = eng.stats()["device_ms"]
        per_it = (ms - short_ms) / max(1, r["pivots"] - short["pivots"]) * 1e3
        packing = len(eng.lower_bound(grid, seed=1)) if len(defs) == 1 else None
        found = [search(eng, grid, defs, weights, s) for s in SEEDS]
        obj = "total weight" if weights else "platforms"
        say(f"{name:38s} certified >= {r['bound']} ({r['pivots']} iterations, {r['constraints']} constraints, {ms:.1f} ms on the device, "
            f"{per_it:.1f} us per iteration; 50 iterations: {short['bound']})"
            + (f"; packing {packing}" if packing is not None else "")
            + f"; search {obj} {found} (mean {np.mean(found):.1f}): gap <= {100 * (min(found) / r['bound'] - 1):.1f} %")
    eng.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
