"""The fractional bound run to optimality on each simplex kernel: LP value reached (total / max load, the certified value with unit
costs), pivots, the optimal flag and device time (median of 5 warm calls), next to the LP optimum from HiGHS (tests/test_lp_reference.py)."""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import timberborn_support_solver_b200 as T
import test_lp_reference as L

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
eng = T.Engine(0)
for grid_name, pset, path in [("ex2", "1x1", "cluster"), ("readme", "1x1", "cluster"), ("rect16", "1x1", "cluster"), ("rect19", "1x1", "cluster"),
                              ("rect21", "1x1", "grid"), ("synth32", "1x1", "grid"), ("rect32", "1x1", "grid"), ("rect32", "default8", "grid"),
                              ("ex2", "1x1", "single"), ("readme", "1x1", "single"), ("rect16", "1x1", "single"), ("rect32", "1x1", "single")]:
    os.environ["TSS_LP_SINGLE_CTA"] = "1" if path == "single" else "0"
    ref = L.reference(grid_name, pset)
    ms = []
    for _ in range(6):
        r = L._lower_bound_lp(eng, grid_name, pset)
        ms.append(eng.stats()["device_ms"])
    v, _ = ref.certified(r["weights"])
    print(json.dumps(dict(case=f"{grid_name}/{pset}", path=path, lp_optimum=round(ref.lp, 9), value=round(float(v), 9), shortfall=round(ref.lp - float(v), 9),
                          bound=r["bound"], pivots=r["pivots"], optimal=r["optimal"], device_ms=round(float(np.median(ms[1:])), 3))), flush=True)
