#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the feasibility-and-bound hot path.

Workload (BASELINE.json configs[1]): rect 16x16 ceiling, 1x1 supports, find the minimum support count.
One "step" = one epoch of the hot path on one GPU: the SLS kernel (b) advances every chain of the portfolio by
`--epoch-steps` steps, the best-reduce kernel folds the chains' best counts into the device-resident bound and (N > 1)
one NCCL all-reduce-min over NVLink shares that bound between the ranks.

Unit (SURVEY.md §8(d)): ONE SLS FLIP — a support added or removed — is one candidate layout evaluated incrementally.
value = flips per second over all ranks, counted by the kernels themselves (tss_stats.sls_flips).  The neighbour layouts a
chain scores to CHOOSE each flip (all k removals, up to 25 additions) are reported beside it, never added to it.
`--impl reference` runs the SAME step rule, the same chains and the same unit on the host cores (oracle/sls_flat.cpp, a
flat-array CPU port that reproduces the kernels' trajectories bit for bit) and never touches the GPU: the reference itself
(Rust + Glucose) cannot be built here, so the CPU arm is the oracle port, on all host threads.

Beside the line, on rank 0 at N = 1: time-to-optimal with the same starting bound on both arms, the REPL's bound-tightening
loop end to end (GPU-seeded against CPU-only), the full-evaluation kernel (a), the CNF kernel (c), the measured
integer-issue / shared-memory peaks, and a bounded CPU baseline.  On every N: the two other multi-GPU configs BASELINE.json
names (C5: the 100k-terrain batch, strong scaling; C4: the 256x256 portfolio, quality at equal phases).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "candidate layouts evaluated/sec"
UNIT = "layouts/s"
WORKLOAD = "rect 16x16 ceiling, 1x1 supports, find minimum support count (BASELINE.json configs[1])"
NO_BOUND = 1 << 20
C4_CHAINS_PER_WINDOW = 16   # configs[3] on both arms (the engine's default for 256x256: more chains per window only slow the steps, profiles/r2_c4_tradeoff.log)
# SURVEY.md §8(d): algorithmic integer work of one flip = one reach-window derivation (7 words x 3 rounds x 5 ops = 105 ops)
# + |R(s)| compare/adds on the cover counters; |R| is measured on the terrain (mean_reach)
A_FLIP_SURVEY = 105
# the kernel's OWN accounting of what it executes per unit (DESIGN.md "kernel (b)"): thread-ops per neighbour layout scored
# and per flip.  Reported as roofline.alu_frac_kernel_ops, i.e. how busy the ALU pipe is, NOT as the algorithmic fraction.
A_SCORE = 7 * 4 + 2      # per candidate scored: 7 window rows x (shift, and, pack, add) + key build
A_FLIP = 7 * 20          # per support added/removed: 7 window rows x (row mask 6 + five-plane add/sub 10 + derive 4)
KERNEL_NAMES = {1: "sls_kernel (one chain per warp)", 2: "sls_h16_kernel (two chains per warp)", 3: "sls_t16_kernel (one chain per thread)",
                4: "sls_p16_kernel (one chain per thread, two grid rows per word)"}
# per-launch DRAM traffic of each variant, PASTED from its committed ncu capture (profiles/): not measured per run
KERNEL_NCU = {
    2: {"traffic": 3067392, "traffic_note": "pasted from profiles/r1_sls_h16_kernel.md (ncu --set full, 9472 chains x 512 steps): chain states only"},
    3: {"traffic": 11063040, "traffic_note": "pasted from profiles/r2_sls_t16_kernel.md (ncu --set full, 56832 chains x 512 steps; dram read 10 978 816 + write 84 224 bytes): chain states + site lists"},
}


def proven_optimum(key):
    """tests/golden/proofs.json: SAT at the optimum and UNSAT one below by the oracle CDCL AND z3 (make_proofs.py)."""
    rec = json.load(open(os.path.join(ROOT, "tests", "golden", "proofs.json")))[key]
    assert rec["proved"]
    return int(rec["optimum"])


OPTIMUM_RECT16 = proven_optimum("rect16/1x1")
C4_NOISE = [20, 12, 28, 8, 35, 16, 24, 5]     # percent of random add moves per rank of the 256x256 portfolio


def workload_config(args):
    """`config` of the JSON line: identical on both arms (the driver compares them)."""
    return {"workload": WORKLOAD,
            "unit_of_work": "one SLS flip (a support added or removed) = one candidate layout evaluated incrementally (SURVEY.md §8(d))",
            "step_rule": "csrc/sls_spec.hpp (min-loss removal, max-gain addition at a random uncovered tile, 20% noise, tabu tenures 3/6/12/20, counter-based RNG); "
                         "chains are seeded (seed 1, global chain index) and reproduce bit for bit on both arms",
            "epoch_steps": args.epoch_steps,
            "l2": "the GPU arm flushes L2 between timed steps (256 MiB memset outside the event pairs); a chain's working set lives in registers / shared memory "
                  "(GPU) or L1/L2 (CPU), HBM / DRAM is touched at epoch start and end only"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_validate_rate(grid, seconds=10.0, threads=None):
    """The reference's own layout check (PlatformLayout::validate, oracle port) on the host cores, bounded sample."""
    import oracle.oracle as O
    threads = threads or os.cpu_count() or 1
    rng = np.random.default_rng(0)
    n = 16384 * threads
    sites = (rng.random((n, grid.shape[0], grid.shape[1])) < 0.06).astype(np.uint8)
    done, t_total = 0, 0.0
    while t_total < seconds:
        _, _, sec = O.validate_sites_batch(grid, sites, threads=threads, flat=True)
        done += n
        t_total += sec
    return done / t_total, threads, (f"{done} random 1x1 layouts (6% density) on rect 16x16 through the oracle's flat-array port of "
                                     f"PlatformLayout::validate, {threads} threads, {t_total:.1f} s")


def cdcl_time_to_optimum(grid, optimum, conflict_budget=400000):
    """Oracle CDCL (Glucose stand-in), 1 thread like the reference (solver_runner.rs:15).
    -> ms of ONE solve handed the bound `optimum` (the same starting bound the GPU arm gets), and ms of the REPL's
    bound-tightening loop from its unbounded first solve until the first layout with `optimum` platforms."""
    import oracle.oracle as O
    cnf = O.Encoding(O.PLATFORMS_1X1, grid).with_limits({(1, 1): optimum})
    r, _, st = cnf.solve(conflict_budget=conflict_budget)
    given = st["seconds"] * 1e3 if r == 10 else None
    loop = O.solver_loop(grid, O.PLATFORMS_1X1, conflict_budget=conflict_budget)
    t, unbounded = 0.0, None
    for s in loop["steps"]:
        t += s["seconds"]
        if s["result"] == 10 and s["count"] <= optimum:
            unbounded = t * 1e3
            break
    return given, unbounded


def cpu_flips(grid, epoch_steps, warm, timed, threads=None, chains_per_thread=32):
    """The SLS step rule on the host cores (oracle/sls_flat.cpp): chains 0.. of seed 1 — the very chains the GPU arm runs —
    `warm` untimed epochs then `timed` epochs.  -> (flips/s over the timed epochs, per-epoch ms, threads, chains, best, sample)"""
    import oracle.oracle as O
    threads = threads or os.cpu_count() or 1
    n = chains_per_thread * threads
    r = O.sls_flat(grid, n, [(epoch_steps, NO_BOUND, 0)] * (warm + timed), seed=1, threads=threads, want_layouts=False)
    sec = float(r["epoch_seconds"][warm:].sum())
    flips = int(r["epoch_flips"][-1]) - (int(r["epoch_flips"][warm - 1]) if warm else 0)
    best = int(r["best"].min())
    sample = (f"{n} chains x {timed} epochs x {epoch_steps} steps of the same step rule and seeds on {threads} host threads "
              f"(oracle/sls_flat.cpp, flat-array port, trajectories identical to the kernels'), {flips} flips in {sec:.2f} s after {warm} warm-up epochs; best count {best}")
    return flips / sec, [float(x) * 1e3 for x in r["epoch_seconds"][warm:]], threads, n, best, sample


def named_grid(fx, name):
    """test/exN.toml from the committed fixtures; "readme" = the README's 21x16 terrain = ex2 with its 2x2 hole filled (SURVEY.md §8d)"""
    rows = fx["ex2" if name == "readme" else name]["grid"]
    w = max(len(r) for r in rows)
    grid = np.array([[1 if (i < len(r) and r[i] == "X") else 0 for i in range(w)] for r in rows], np.uint8)
    if name == "readme":
        grid[8:10, 8:10] = 1
    return grid


def repl_loop_cpu(name_defs):
    """crates/repl/src/main.rs:280-366 on the CPU alone (oracle encoder + CDCL stand-in, 1 thread): wall ms per instance."""
    import oracle.oracle as O
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "fixtures.json")))
    out = {}
    for name, label in name_defs:
        grid = named_grid(fx, name)
        t0 = time.perf_counter()
        r = O.solver_loop(grid, O.PLATFORMS_DEFAULT if label == "default-8" else O.PLATFORMS_1X1, conflict_budget=20_000_000)
        ms = (time.perf_counter() - t0) * 1e3
        out[f"{name} {label}"] = {"ms": ms, "solves": len(r["steps"]), "optimum": len(r["best"]), "proved": bool(r["proved_optimal"])}
    return out


REPL_INSTANCES = [("ex1", "default-8"), ("ex3", "default-8"), ("ex2", "default-8"), ("ex2", "1x1"), ("readme", "1x1")]


def synthetic_terrain(w, h, t=0, seed=1):
    """SURVEY.md §8(d): ceiling iff (splitmix64(seed * 0x9E3779B97F4A7C15 + (t << 20) + y * w + x) >> 40) < floor(0.7 * 2^24) — the
    generator of configs[3] / configs[4], restated here so that the CPU arm needs nothing of the product."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + np.arange(w * h, dtype=np.uint64) + (np.uint64(t) << np.uint64(20))
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return ((z >> np.uint64(40)) < np.uint64(11744051)).astype(np.uint8).reshape(h, w)


def c5_reference(steps):
    """configs[4] on the CPU arm: a bounded sample of the batch's first terrains."""
    n = 32 * (os.cpu_count() or 1)
    grids = np.stack([synthetic_terrain(32, 32, t) for t in range(n)])
    return c5_cpu_sample(grids, 0, steps)[1]


def c4_cpu_sample(grid, chains_per_window, phase_steps, phases=2):
    """configs[3] on the host cores: the window decomposition's scalar replay with the chains through the flat-array port
    (oracle.lns_model(flat=True): same windows, chains, seeds and step rule as csrc/lns.cu), one window per worker thread, for the
    first `phases` phases from the all-supports start layout.  -> (counts after every phase, dict for the JSON line)"""
    import oracle.oracle as O
    threads = os.cpu_count() or 1
    st = {}
    t0 = time.perf_counter()
    res = O.lns_model(grid, chains_per_window, phases, phase_steps, seed=1, flat=True, threads=threads, stats=st)
    wall = time.perf_counter() - t0
    counts = [c for _, c in res]
    return counts, {"flips_per_s": st["flips"] / st["seconds"], "cores": threads, "kind": "port", "counts": counts, "ms_per_phase": wall * 1e3 / phases,
                    "sample": f"the first {phases} phases x {phase_steps} steps of the 256x256 search from the all-supports layout, {chains_per_window} chains per window "
                              f"(oracle.lns_model + oracle/sls_flat.cpp, same windows / chains / seeds as the GPU arm), one window per host thread, {wall:.1f} s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    grid = np.ones((16, 16), np.uint8)
    W, K = max(args.warmup, 3), args.steps
    value, epoch_ms, threads, n_chains, best, sample = cpu_flips(grid, args.epoch_steps, W, K)
    given, unbounded = cdcl_time_to_optimum(grid, OPTIMUM_RECT16)
    vrate, vthreads, vsample = cpu_validate_rate(grid, seconds=3.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": float(np.mean(epoch_ms)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 bitboards / bool",
        "data": "synthetic", "config": workload_config(args),
        "run": {"chains": n_chains, "threads": threads, "note": "reference = CPU path; the reference's own code (Rust + rustsat-glucose) cannot be built here, so this arm is the oracle port"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "best_count": best,
        "time_to_optimal_ms": given,
        "time_to_optimal": {"given_bound_ms": given, "from_unbounded_ms": unbounded, "optimum": OPTIMUM_RECT16,
                            "note": "oracle CDCL (Glucose stand-in), 1 solver thread as in the reference (solver_runner.rs:15): one solve handed the bound 15 / the REPL loop "
                                    "from its unbounded first solve to the first layout with 15 supports; the UNSAT proof of 14 (minutes, tests/golden/proofs.json) is not included"},
        "repl_loop": repl_loop_cpu(REPL_INSTANCES),
        "validate_layouts_per_s": vrate, "validate_sample": vsample,
        "other_configs": {"c5": c5_reference(2000), "c4": c4_cpu_sample(synthetic_terrain(256, 256), C4_CHAINS_PER_WINDOW, args.phase_steps)[1]},
    }
    print(json.dumps(line), flush=True)


def setup_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the GPU path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return torch, dist, world, rank, local


def comm_init(eng, torch, dist, rank, world):
    """The engine's own NCCL communicator: torch.distributed only carries the 128-byte id."""
    idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(eng.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(idt, src=0)
    eng.comm_init(bytes(idt.cpu().numpy().tobytes()), rank, world)


def run_c5(args):
    """BASELINE.json configs[4]: batch of 100k synthetic 32x32 terrains (p = 0.7), contiguous shards per GPU, no data-path
    collective; one all-gather of the per-terrain counts at the end.  A step = one pass over the whole batch."""
    import ctypes as C
    torch, dist, world, rank, local = setup_dist()
    import timberborn_support_solver_b200 as T
    eng = T.Engine(local)
    from timberborn_support_solver_b200.portfolio import shard_range
    n_total = args.terrains
    lo, hi = shard_range(n_total, rank, world)
    lib = T.load()
    grids = np.zeros((hi - lo, 32, 32), np.uint8)
    for i, t in enumerate(range(lo, hi)):
        lib.tss_world_synthetic(32, 32, 1, t, int(0.7 * (1 << 24)), grids[i].ctypes.data_as(C.POINTER(C.c_uint8)))
    W, K = max(args.warmup, 1), args.steps
    for _ in range(W):
        eng.solve_batch(grids[: min(len(grids), 8192)], seed=1, steps=args.batch_steps)
    sampler = ClockSampler(local)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    s0 = eng.stats()
    dev_ms, t0 = 0.0, time.perf_counter()
    for _ in range(K):
        counts, layouts = eng.solve_batch(grids, seed=1, steps=args.batch_steps, want_layouts=True)
        dev_ms += eng.stats()["device_ms"]
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    s1 = eng.stats()
    sampler.stop_flag = True
    sampler.join()
    # final gather: 4 bytes per terrain
    cd = torch.from_numpy(counts).cuda()
    if world > 1:
        sizes = [shard_range(n_total, r, world)[1] - shard_range(n_total, r, world)[0] for r in range(world)]
        parts = [torch.empty(sz, dtype=torch.int32, device="cuda") for sz in sizes]
        dist.all_gather(parts, cd)
        allc = torch.cat(parts)
    else:
        allc = cd
    tt = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(s1["candidates_scored"] - s0["candidates_scored"]), float(s1["kernel_launches"] - s0["kernel_launches"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    if rank == 0:
        dev_ms_max, wall_ms_max = (float(x) for x in tt.tolist())
        tiles = grids.reshape(len(grids), -1).sum(1)
        # every reported layout of rank 0's shard re-evaluated by kernel (a) in per-terrain mode: complete, count matches
        terr_rows = (grids.astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(2, dtype=np.uint32)
        g_dev, l_dev = torch.from_numpy(terr_rows.view(np.int32)).cuda(), torch.from_numpy(layouts.view(np.int32)).cuda()
        out = torch.empty((len(grids), 2), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        eng.eval_compact_dev(g_dev.data_ptr(), 32, 32, l_dev.data_ptr(), len(grids), out.data_ptr(), per_layout_terrain=True)
        torch.cuda.synchronize()
        res = out.cpu().numpy()
        ok = bool((res[:, 0] == 0).all() and np.array_equal(res[:, 1], counts))
        line = {"metric": "terrains solved/sec (per-terrain best support count)", "value": n_total * K / (dev_ms_max * 1e-3), "unit": "terrains/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms_max / K, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u32 bitboards / bool", "data": "synthetic",
                "config": {"workload": f"batch of {n_total} synthetic 32x32 terrains (p=0.7), 1x1 supports (BASELINE.json configs[4])", "sls_steps_per_chain": args.batch_steps,
                           "chains_per_terrain": 4, "parallelism": f"terrain shards x{world}, no data-path collective, final all-gather of counts",
                           "l2": "inputs larger than L2 (100 MB of terrains, 800 MB of reach tables per pass)"},
                "e2e": {"value": n_total * K / (wall_ms_max * 1e-3), "unit": "terrains/s", "h2d_bytes_per_step": int(grids.size), "d2h_bytes_per_step": int(counts.nbytes + layouts.nbytes),
                        "note": "tss_solve_batch from host u8 grids to host counts + layouts, wall clock, slowest rank"},
                "gpu_launches": int(tot[1].item()), "candidates_per_s": float(tot[0].item()) / (dev_ms_max * 1e-3), "mean_count": float(allc.float().mean().item()),
                "mean_ceiling_tiles": float(tiles.mean()), "witnesses_revalidated_by_kernel_a": ok, "clocks": sampler.summary(),
                }
        if world == 1:
            # bounded CPU baseline: the reference's loop (oracle CDCL as the Glucose stand-in, 1 thread per instance like the
            # reference) on the first terrains of the batch, a conflict budget per solve instead of minutes per terrain
            import oracle.oracle as O
            t0 = time.perf_counter()
            cpu_counts = []
            for t in range(2):
                r = O.solver_loop(grids[t], O.PLATFORMS_1X1, conflict_budget=50000)
                cpu_counts.append(min(s["count"] for s in r["steps"] if s["result"] == 10))
            cpu_s = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": 2 / cpu_s, "unit": "terrains/s", "cores": 1, "kind": "port",
                                    "sample": f"terrains 0-1 of the batch through the oracle's CDCL bound-tightening loop, 50000 conflicts per solve, {cpu_s:.1f} s: "
                                              f"counts {cpu_counts} (unproven), GPU counts for the same terrains {[int(c) for c in counts[:2]]}"}
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def run_c4(args):
    """BASELINE.json configs[3]: synthetic 256x256 ceiling (p = 0.7), window-decomposed SLS portfolio, one seed set per GPU,
    all-reduce-min of (count, rank) + the winner's layout after every phase.  A step = one phase."""
    torch, dist, world, rank, local = setup_dist()
    import timberborn_support_solver_b200 as T
    eng = T.Engine(local)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    if world > 1:
        comm_init(eng, torch, dist, rank, world)
    g = T.WorldGrid.synthetic(256, 256, 1, 0)
    s = eng.search(g, seed=1, n_chains=args.chains, chain_offset=rank * 1000000, noise_pct=C4_NOISE[rank % len(C4_NOISE)])     # 0 = one wave of chains over the windows
    W, K = max(args.warmup, 3), args.steps
    for _ in range(W):
        s.run(args.phase_steps, 0)
    s.best_count()
    s0 = eng.stats()
    sampler = ClockSampler(local)
    sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    for a, b in evs:
        a.record()
        s.run(args.phase_steps, 0)
        b.record()
    torch.cuda.synchronize()
    count = s.global_best()
    s1 = eng.stats()
    sampler.stop_flag = True
    sampler.join()
    lay = s.best_layout()            # re-validated by kernel (a) inside the engine
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    # e2e: the same terrain through the one-shot C-ABI call with HOST buffers on every rank (workspace creation, terrain
    # upload, K phases, layout download + validation inside the timed region)
    e0 = eng.stats()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    res, lay_e2e = eng.solve_upper_bound(g, card_limit=None, seed=50 + rank, max_steps=K * args.phase_steps)
    t_e2e = time.perf_counter() - t0
    e1 = eng.stats()
    e2e_t = torch.tensor([float(e1["sls_flips"] - e0["sls_flips"]), t_e2e], dtype=torch.float64, device="cuda")
    e2e_max = e2e_t.clone()
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.SUM)
        dist.all_reduce(e2e_max, op=dist.ReduceOp.MAX)
    tt = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(s1["sls_flips"] - s0["sls_flips"]), float(s1["kernel_launches"] - s0["kernel_launches"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    if rank == 0:
        ms = float(tt.item())
        line = {"metric": METRIC, "value": float(tot[0].item()) / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 bitboards / bool", "data": "synthetic",
                "config": {"workload": "synthetic 256x256 random ceiling mask (density 0.7), 1x1 supports, SLS portfolio with all-reduce-min bound (BASELINE.json configs[3])",
                           "phase_steps": args.phase_steps, "chains_total": s.n_chains, "parallelism": f"portfolio x{world}: window decomposition per GPU, winner's layout shipped after every phase"},
                "gpu_launches": int(tot[1].item()), "best_count": count, "layout_platforms": lay.platform_count(), "ceiling_tiles": int(g.data.sum()),
                "phases_total": W + K, "clocks": sampler.summary(),
                "e2e": {"value": float(e2e_t[0].item()) / float(e2e_max[1].item()), "unit": UNIT, "h2d_bytes_per_step": int(g.data.size // max(K, 1)),
                        "d2h_bytes_per_step": int(20 * lay_e2e.platform_count() // max(K, 1)), "count": lay_e2e.platform_count(),
                        "note": f"tss_solve_upper_bound from a host u8 grid to a host platform list on each of the {world} rank(s): workspace creation, upload, "
                                f"{K} phases of {args.phase_steps} steps, layout download and validation; wall clock, sum over ranks / slowest rank"}}
        print(json.dumps(line), flush=True)
    s.close()
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def c5_cpu_sample(grids, first_terrain, steps, n_sample=None):
    """BASELINE.json configs[4] on the host cores: the same four chains per terrain, seeds and step rule as tss_solve_batch (chains
    4t .. 4t+3 of seed 1, the bound shared every 1024 steps) through the oracle's flat-array port, one terrain per worker thread.
    -> (counts of the sample, dict for the JSON line)"""
    import oracle.oracle as O
    from concurrent.futures import ThreadPoolExecutor
    threads = os.cpu_count() or 1
    n_sample = min(len(grids), n_sample or 32 * threads)
    epochs = [(min(1024, steps - d), NO_BOUND, 0) for d in range(0, steps, 1024)]

    def one(i):
        r = O.sls_flat(grids[i], 4, epochs, seed=1, chain_offset=4 * (first_terrain + i), threads=1, want_layouts=False)
        return int(r["best"].min())
    one(0)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        counts = list(ex.map(one, range(n_sample)))
    sec = time.perf_counter() - t0
    return counts, {"terrains_per_s": n_sample / sec, "cores": threads, "kind": "port",
                    "sample": f"terrains {first_terrain}..{first_terrain + n_sample - 1} of the batch, 4 chains x {steps} steps each (oracle/sls_flat.cpp, same chains and seeds as the GPU batch), "
                              f"one terrain per host thread, {sec:.2f} s", "mean_count": float(np.mean(counts))}


def side_c5(eng, torch, dist, world, rank, n_total, steps):
    """BASELINE.json configs[4] at this N (strong scaling: the batch is fixed, ranks take contiguous shards, no data-path
    collective): device time of one pass with the shard's terrains resident in HBM, and the same through tss_solve_batch from
    host buffers.  Returns the dict rank 0 reports (None elsewhere)."""
    import ctypes as C
    import timberborn_support_solver_b200 as T
    from timberborn_support_solver_b200.portfolio import shard_range
    lib = T.load()
    lo, hi = shard_range(n_total, rank, world)          # contiguous, balanced ranges of terrains (SURVEY.md §8e)
    grids = np.zeros((hi - lo, 32, 32), np.uint8)
    for i, t in enumerate(range(lo, hi)):
        lib.tss_world_synthetic(32, 32, 1, t, int(0.7 * (1 << 24)), grids[i].ctypes.data_as(C.POINTER(C.c_uint8)))
    eng.solve_batch(grids[: min(len(grids), 32768)], seed=1, steps=64)              # workspace allocation (one full chunk) + warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    counts = eng.solve_batch(grids, seed=1, steps=steps)
    wall = time.perf_counter() - t0
    dev_ms = eng.stats()["device_ms"]
    t = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device="cuda")
    acc = torch.tensor([float(counts.sum()), float(len(counts))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    if rank != 0:
        return None
    gap = None
    if world == 1:      # how far from optimal are the counts?  certified lower bounds on a sample (the exact solver cannot finish a terrain in minutes)
        sample = range(0, 32)
        lbs = [max(len(eng.lower_bound(T.WorldGrid(grids[i]), seed=1)), eng.lower_bound_lp(T.WorldGrid(grids[i]))["bound"]) for i in sample]
        gap = {"terrains": len(lbs), "mean_count": float(np.mean([counts[i] for i in sample])), "mean_certified_lower_bound": float(np.mean(lbs)),
               "max_gap": int(max(int(counts[i]) - lb for i, lb in zip(sample, lbs))), "min_gap": int(min(int(counts[i]) - lb for i, lb in zip(sample, lbs))),
               "proven_optimal": int(sum(1 for i, lb in zip(sample, lbs) if int(counts[i]) == lb)),
               "note": "terrains 0-31 of the batch: SLS count against max(packing bound, fractional LP bound), both certified on the GPU (tss_lower_bound, tss_lower_bound_lp)"}
    dev_ms_max, wall_ms_max = (float(x) for x in t.tolist())
    cpu = None
    if world == 1:      # the same chains on the host cores, a bounded sample: terrains/s beside the GPU's, and the counts must be the same numbers
        cpu_counts, cpu = c5_cpu_sample(grids, lo, steps)
        cpu["counts_identical_to_gpu"] = bool(all(int(counts[i]) == c for i, c in enumerate(cpu_counts)))
    return {"optimality_gap_sample": gap, "cpu_baseline": cpu, "workload": f"batch of {n_total} synthetic 32x32 terrains (p=0.7), 1x1 supports, {steps} SLS steps per chain (BASELINE.json configs[4])",
            "scaling": "strong", "terrains_per_s": n_total / (dev_ms_max * 1e-3), "ms": dev_ms_max,
            "e2e": {"terrains_per_s": n_total / (wall_ms_max * 1e-3), "ms": wall_ms_max, "h2d_bytes": int(n_total * 1024), "d2h_bytes": int(n_total * 4),
                    "note": "tss_solve_batch from host u8 grids to host counts, wall clock, slowest rank"},
            "mean_count": float(acc[0].item() / acc[1].item()), "terrains": int(acc[1].item())}


def side_c4(eng, torch, dist, world, rank, phases, phase_steps):
    """BASELINE.json configs[3] at this N: 256x256 window-decomposed portfolio, every rank its own seeds, per-window best of all
    ranks combined after every phase.  Quality at equal phases (= equal time: per-rank work does not depend on N)."""
    import timberborn_support_solver_b200 as T
    g = T.WorldGrid.synthetic(256, 256, 1, 0)
    # diversification by rank, not just other seeds: every rank searches with its own noise level (rank 0: the default 20 %), and
    # the per-window combination keeps, window by window, whatever worked best
    s = eng.search(g, seed=1, n_chains=C4_CHAINS_PER_WINDOW, chain_offset=rank * 1000000, noise_pct=C4_NOISE[rank % len(C4_NOISE)])
    s.run(phase_steps, 0)                  # warm-up phase (allocations, first descent from the all-supports layout)
    s.best_count()
    f0 = eng.stats()
    evs = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    evs[0].record()
    for _ in range(phases):
        s.run(phase_steps, 0)
    evs[1].record()
    torch.cuda.synchronize()
    count = s.global_best()
    f1 = eng.stats()
    lay = s.best_layout()                  # re-validated by kernel (a) inside the engine
    assert lay.platform_count() == count
    lower = len(eng.lower_bound(g, seed=1)) if rank == 0 else 0     # certified packing bound (whole-board rounds, csrc/lb.cu)
    lower_ms = eng.stats()["device_ms"]
    t = torch.tensor([evs[0].elapsed_time(evs[1])], dtype=torch.float64, device="cuda")
    acc = torch.tensor([float(f1["sls_flips"] - f0["sls_flips"]), float(f1["candidates_scored"] - f0["candidates_scored"])], dtype=torch.float64, device="cuda")
    cmin = torch.tensor([float(count)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        dist.all_reduce(cmin, op=dist.ReduceOp.MIN)
    n_chains = s.n_chains
    s.close()
    cpu = None
    if world == 1:   # the same first two phases on the host cores (bounded sample): flips/s beside the GPU's, and the counts must be the same numbers
        per_window = n_chains // 81
        s2 = eng.search(g, seed=1, n_chains=per_window)
        gpu_counts = []
        for _ in range(2):
            s2.run(phase_steps, 0)
            gpu_counts.append(int(s2.best_count()))
        s2.close()
        cpu_counts, cpu = c4_cpu_sample(g.data, per_window, phase_steps)
        cpu["counts_identical_to_gpu"] = bool(cpu_counts == gpu_counts)
    if rank != 0:
        return None
    ms = float(t.item())
    return {"workload": "synthetic 256x256 random ceiling (p=0.7), 1x1 supports, window-decomposed SLS portfolio (BASELINE.json configs[3])",
            "scaling": "weak (own seeds and noise level per rank; per-window best of all ranks adopted after every phase)", "best_count": int(cmin.item()),
            "ceiling_tiles": int(g.data.sum()), "certified_lower_bound": lower, "lower_bound_ms": lower_ms, "cpu_baseline": cpu,
            "trivial_lower_bound": int(-(-int(g.data.sum()) // 25)), "phases": phases + 1, "phase_steps": phase_steps,
            "ms": ms, "flips_per_s": float(acc[0].item()) / (ms * 1e-3), "neighbour_scores_per_s": float(acc[1].item()) / (ms * 1e-3), "chains_per_gpu": n_chains}


def repl_loop_cpp_driver(name_defs):
    """The same loop through the C++ driver over the C ABI (timberborn_support_solver_b200/tss_repl = tools/tss_repl.cpp: the Rust
    shim's call sequence, tss_cnf_upload -> tss_instance_find -> tss_solve_instance, no exact solver attached): one whole
    `load; solve` repeated 21 times in one process, warm median wall ms (engine creation = CUDA context start-up excluded)."""
    import re
    import subprocess
    import tempfile
    import timberborn_support_solver_b200 as T
    exe = os.path.join(os.path.dirname(T.__file__), "tss_repl")
    if not os.path.exists(exe):
        return {"unavailable": "tss_repl not built (python -m timberborn_support_solver_b200.build)"}
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "fixtures.json")))
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, label in name_defs:
            path = os.path.join(tmp, f"{name}.toml")
            with open(path, "w") as f:
                f.write(T.WorldGrid(named_grid(fx, name)).to_toml())
            r = subprocess.run([exe, path, "--platforms", "default" if label == "default-8" else "1x1", "--seed", "3", "--quiet", "--repeat", "21"],
                               capture_output=True, text=True, timeout=300)
            m = re.search(r'# best=(\d+) lower_bound=(-?\d+) verdict="([^"]*)" gpu_solves=(\d+) exact_solves=(\d+) ms=([\d.]+) setup_ms=([\d.]+) repeats=\d+ warm_ms=([\d.]+)', r.stdout)
            out[f"{name} {label}"] = ({"warm_ms": float(m.group(8)), "cold_ms": float(m.group(6)), "optimum": int(m.group(1)), "verdict": m.group(3),
                                       "gpu_solves": int(m.group(4)), "exact_solves": int(m.group(5))} if r.returncode == 0 and m else {"error": (r.stderr or r.stdout)[-200:]})
    return out


def oracle_exact(cnf):
    """The exact solver of the REPL loop (rustsat-glucose in the reference; here the oracle's CDCL stand-in, as on the CPU arm)."""
    import ctypes as C
    import oracle.oracle as O
    import timberborn_support_solver_b200 as T
    a = np.full(cnf.n_vars + 1, 2, np.uint8)
    lits, offs = np.ascontiguousarray(cnf.lits, np.int32), np.ascontiguousarray(cnf.offsets, np.uint32)
    r = O.lib().tsso_solve_csr(O._p(lits), O._p(offs, C.c_uint32), cnf.n_clauses, cnf.n_vars, O._p(a, C.c_uint8), C.c_long(-1))
    return {10: T.SAT, 20: T.UNSAT}.get(r, T.INTERRUPTED), a


def repl_loop_gpu(eng, name_defs):
    """crates/repl/src/main.rs:280-366 with the GPU engine answering the SAT iterations (and its certified lower bounds — integral
    packing, then the fractional LP — ending the loop when they meet the count) and the exact solver called only for what is
    left: wall ms per instance to the PROVEN optimum, host buffers."""
    import timberborn_support_solver_b200 as T
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "fixtures.json")))
    out = {}
    for name, label in name_defs:
        grid = T.WorldGrid(named_grid(fx, name))
        defs = T.PLATFORMS_DEFAULT if label == "default-8" else T.PLATFORMS_DEFAULT[:1]
        ts, res = [], None
        for rep in range(3):
            t0 = time.perf_counter()
            enc = T.Encoding.encode(defs, grid)
            res = T.solver_loop(T.Project(T.World(grid)), enc, T.PlatformLimits(), eng, exact_solver=oracle_exact, seed=rep)
            ts.append((time.perf_counter() - t0) * 1e3)
        out[f"{name} {label}"] = {"ms": float(min(ts)), "gpu_solves": sum(1 for st in res["steps"] if st["source"] == "gpu"),
                                  "exact_solves": sum(1 for st in res["steps"] if st["source"] == "exact"), "optimum": res["best"].platform_count(),
                                  "proved": bool(res["proved_optimal"]), "lower_bound": res.get("lower_bound")}
    return out


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, search):
    """What the timed path hands its caller after the last timed step, one float64 DIR/<name>.npy per array (exact for every
    integer it holds): each chain's current and best support rows (one word per grid row, bit x = column x), support count, best
    count, step and score counters, and the portfolio's best count and best layout (x, y, def_w, def_h, rotated; row-major order).
    Beyond DUMP_BYTES in all, a fixed sample of the chains (seed 0) is written; chain_index names the chains of every chain_* file."""
    st = search.read_chains()
    h = search.grid.height
    chains = {"chain_supports": st["S"][:, :h], "chain_best_supports": st["bestS"][:, :h], "chain_count": st["k"], "chain_best_count": st["best"],
              "chain_step": st["step"], "chain_scored": st["scored"], "chain_index": np.arange(search.n_chains)}
    per_chain = 8 * sum(a[0].size for a in chains.values())
    keep = (DUMP_BYTES - (1 << 20)) // per_chain        # 1 MiB left for the best layout, the best count and the .npy headers
    if search.n_chains > keep:
        idx = np.sort(np.random.default_rng(0).choice(search.n_chains, keep, replace=False))
        chains = {k: v[idx] for k, v in chains.items()}
    best = search.best_count()
    layout = [] if best is None else sorted(((p.x, p.y, p.definition.width, p.definition.height, int(p.rotated))
                                             for p in search.best_layout().platforms().values()), key=lambda p: (p[1], p[0]))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in dict(chains, best_count=[-1 if best is None else best], best_layout=np.reshape(layout, (-1, 5))).items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--epoch-steps", type=int, default=4096, help="SLS steps per chain per bench step")
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (0 = fill the device for the chosen kernel)")
    ap.add_argument("--kernel", type=int, default=0, help="SLS kernel variant (tss.h TSS_KERNEL_*: 0 auto, 1 warp, 2 half-warp, 3 thread, 4 thread / row pairs)")
    ap.add_argument("--quick", action="store_true", help="skip the side measurements (peaks, eval/cnf kernels, other configs, cpu baseline)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c4", "c5"], help="c2 = the bench line (rect 16x16); c4 / c5 = the other named configs on their own")
    ap.add_argument("--terrains", type=int, default=100000, help="c5: terrains in the batch")
    ap.add_argument("--batch-steps", type=int, default=2000, help="c5: SLS steps per chain")
    ap.add_argument("--phase-steps", type=int, default=4000, help="c4: SLS steps per window-decomposition phase")
    ap.add_argument("--c4-phases", type=int, default=15, help="c4 side measurement of the default line: timed phases")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (rank 0's chains, the best count "
                                                          "and layout) as DIR/<name>.npy, float64, at most 64 MB (c2 on the GPU arm)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "c2"):
        ap.error("--dump-outputs: only the c2 workload on the GPU arm")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "c5":
        return run_c5(args)
    if args.workload == "c4":
        return run_c4(args)

    import torch
    import torch.distributed as dist

    import timberborn_support_solver_b200 as T

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the GPU path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = max(args.warmup, 3)
    K = args.steps

    eng = T.Engine(local)
    # torch events only see torch's current stream: make one explicit (non-default) stream current and hand it to the
    # engine, so every kernel of the hot path and every event of this file live on the same stream
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)
    info = eng.device_info()
    grid = T.WorldGrid(np.ones((16, 16), np.uint8))
    exchange = "none (single GPU)"
    if world > 1:
        # the path's one real exchange: an all-reduce-min of the best-known count (4 bytes, latency bound).  The engine does
        # it itself, in-stream on the device-resident bound (ncclAllReduce inside tss_search_run); torch.distributed only
        # carries the 128-byte NCCL id from rank 0 to the other ranks.
        comm_init(eng, torch, dist, rank, world)
        exchange = "ncclAllReduce(min, 1 x int32) in-stream inside tss_search_run, bound stays in HBM"
    n_chains = args.chains
    if not n_chains:                 # engine default: fills the device for the chosen kernel
        probe = eng.search(grid, kernel=args.kernel)
        n_chains = probe.n_chains
        probe.close()
    search = eng.search(grid, seed=1, n_chains=n_chains, chain_offset=rank * n_chains, kernel=args.kernel)
    variant = search.kernel_variant()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def step():
        search.run(args.epoch_steps, 0)

    # mean |R(s)| of the terrain (SURVEY.md §8d asks for it beside the rate): one-support layouts through kernel (a)
    one_hot = np.eye(grid.data.size, dtype=np.uint8).reshape(-1, grid.height, grid.width)
    unc1, _ = eng.eval_sites(grid, one_hot)
    mean_reach = float((int(grid.data.sum()) - unc1[grid.data.reshape(-1) != 0]).mean())
    for _ in range(W):
        step()
    search.best_count()        # synchronises and folds the warm-up's device counters into the stats BEFORE the baseline snapshot
    torch.cuda.synchronize()
    s0 = eng.stats()
    sampler = ClockSampler(local)
    sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    for a, b in evs:
        flush.zero_()                       # L2 flush between timed iterations (outside the event pair)
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall = time.perf_counter() - t_wall0
    sampler.stop_flag = True
    sampler.join()
    best = search.best_count()
    s1 = eng.stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, search)
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    tot = torch.tensor([float(s1[k] - s0[k]) for k in ("sls_flips", "candidates_scored", "sls_steps", "kernel_launches")], dtype=torch.float64, device="cuda")
    tmax = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    flips_all, scored_all, steps_all, launches_all = (float(x) for x in tot.tolist())
    ms_total = float(tmax.item())
    sec = ms_total * 1e-3
    value = flips_all / sec

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_total / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 bitboards / bool", "data": "synthetic",
        "config": workload_config(args),
        "run": {"chains_per_gpu": n_chains, "kernel": KERNEL_NAMES.get(variant, str(variant)), "parallelism": f"portfolio x{world} (independent seeds, all-reduce-min of the bound per step)", "exchange": exchange},
        "gpu_launches": int(launches_all), "best_count": best, "proven_optimum": OPTIMUM_RECT16,
        "sls_steps_per_s": steps_all / sec, "flips_per_step": flips_all / max(steps_all, 1.0),
        "neighbour_scores_per_s": scored_all / sec, "neighbour_scores_per_flip": scored_all / max(flips_all, 1.0), "mean_reach": mean_reach,
        "wall_ms_total": t_wall * 1e3, "clocks": sampler.summary(),
    }

    if rank == 0:
        # ---------------- roofline of the dominant kernel (SLS) against the measured LOP3 issue peak.
        # achieved / frac: SURVEY.md §8(d)'s ALGORITHMIC work — (105 + |R|) integer ops per flip — per second.  The search
        # rule (score every removal and every addition in reach before each flip) executes far more than that:
        # alu_frac_kernel_ops is the kernel's own op count over the same peak, i.e. how busy the ALU pipe is.
        pk = eng.measure_peaks()
        a_flip = A_FLIP_SURVEY + mean_reach
        achieved = flips_all * a_flip / sec / 1e9 / world
        kernel_ops = (A_SCORE * scored_all + A_FLIP * flips_all) / sec / 1e9 / world
        ncu = KERNEL_NCU.get(variant, {"traffic": None, "traffic_note": "no ncu capture pasted for this variant"})
        line["roofline"] = {"bound": "int_issue", "achieved": achieved, "peak": pk["lop3_gops"], "unit": "Gop/s", "frac": achieved / pk["lop3_gops"],
                            "traffic": ncu["traffic"], "traffic_note": ncu["traffic_note"], "kernel": KERNEL_NAMES.get(variant, str(variant)),
                            "algorithmic_ops": f"SURVEY.md §8(d): A_flip = 105 + |R| = {a_flip:.1f} integer ops per flip (|R| = mean_reach), flips counted by the kernel",
                            "alu_frac_kernel_ops": kernel_ops / pk["lop3_gops"],
                            "kernel_ops": f"{A_SCORE} thread-ops per neighbour layout scored + {A_FLIP} per flip (DESIGN.md kernel (b)): what the step rule executes, = ALU pipe utilisation",
                            "peak_source": "measured in this run (tss_measure_peaks: dependent-free LOP3 chains at full occupancy)",
                            "note": "no dense contraction and ~0 HBM traffic in the step loop: the bound is integer issue (SURVEY.md §8d); per-GPU figures"}
        line["measured_peaks"] = pk
    # ---------------- e2e through the C ABI with HOST buffers (grid in, layout out) on every rank at once: a fixed step budget
    # per call; terrain upload, reach table, epochs with their host round trips, witness validation and the layout copy back
    # are all inside the timed region.  Whole-job value = flips of all ranks / slowest rank's wall time.
    steps_per_call, n_calls = 16384, 5
    eng.solve_upper_bound(grid, card_limit=None, seed=199, max_steps=steps_per_call)      # workspace warm-up (allocation)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0 = eng.stats()
    t0 = time.perf_counter()
    for i in range(n_calls):
        res, lay = eng.solve_upper_bound(grid, card_limit=None, seed=200 + 16 * rank + i, max_steps=steps_per_call)
    t_e2e = time.perf_counter() - t0
    e1 = eng.stats()
    e2e_t = torch.tensor([float(e1["sls_flips"] - e0["sls_flips"]), t_e2e], dtype=torch.float64, device="cuda")
    e2e_max = e2e_t.clone()
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.SUM)
        dist.all_reduce(e2e_max, op=dist.ReduceOp.MAX)
    line["e2e"] = {"value": float(e2e_t[0].item()) / float(e2e_max[1].item()), "unit": UNIT,
                   "h2d_bytes_per_step": int(grid.data.size + 8), "d2h_bytes_per_step": int(20 * lay.platform_count() + 16 * 9 + 288),
                   "note": f"tss_solve_upper_bound from a host u8 grid to a host platform list on each of the {world} rank(s), {steps_per_call} steps/chain per call, "
                           f"{n_calls} calls, wall clock incl. copies, epoch round trips and witness validation; sum over ranks / slowest rank"}
    search.close()
    # ---------------- the two other multi-GPU configs BASELINE.json names, on EVERY N (all ranks take part)
    if not args.quick:
        others = {}
        c5 = side_c5(eng, torch, dist, world, rank, args.terrains, args.batch_steps)
        c4 = side_c4(eng, torch, dist, world, rank, args.c4_phases, args.phase_steps)
        if rank == 0:
            others["c5"], others["c4"] = c5, c4
            line["other_configs"] = others
    if rank == 0:
        # ---------------- time-to-optimal, both starting points (per rank, identical at every N: a one-shot solve never communicates)
        tto = []
        for seed in range(7):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res, lay = eng.solve_upper_bound(grid, card_limit=OPTIMUM_RECT16, seed=100 + seed)
            tto.append((time.perf_counter() - t0) * 1e3)
            assert res == T.SAT and lay.platform_count() == OPTIMUM_RECT16
        tun = []
        for seed in range(5):                # the REPL schedule: first solve unbounded, then bound = found - 1 (main.rs:346), until 15 is on the table
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            limit, count = None, None
            while count is None or count > OPTIMUM_RECT16:
                res, lay = eng.solve_upper_bound(grid, card_limit=limit, seed=300 + seed)
                assert res == T.SAT
                count = lay.platform_count()
                limit = count - 1
            tun.append((time.perf_counter() - t0) * 1e3)
        line["time_to_optimal_ms"] = float(np.median(tto[2:]))
        line["time_to_optimal"] = {"given_bound_ms": float(np.median(tto[2:])), "from_unbounded_ms": float(np.median(tun[1:])), "optimum": OPTIMUM_RECT16,
                                   "note": "tss_solve_upper_bound from host buffers on one GPU (terrain upload, reach table, fused first epoch, witness re-validated by kernel (a)): "
                                           "one call handed the bound 15 (median of 5 after 2 warm-up calls) / the REPL schedule from an unbounded first call, bound = found - 1, "
                                           "until a layout with 15 supports (median of 4 after 1 warm-up run); same two starting points as the CPU arm"}
    if rank == 0 and not args.quick and world == 1:
        hbm_peak, hbm_src = peaks()
        # ---------------- kernel (a): stream 4 Mi candidate layouts (32 B each, 128 MiB > L2) from HBM
        n_lay = 4 << 20
        lay_dev = torch.randint(0, 1 << 16, (n_lay, 16), dtype=torch.int32, device="cuda")
        lay_dev = (lay_dev & torch.randint(0, 1 << 16, (n_lay, 16), dtype=torch.int32, device="cuda") & torch.randint(0, 1 << 16, (n_lay, 16), dtype=torch.int32, device="cuda")
                   & torch.randint(0, 1 << 16, (n_lay, 16), dtype=torch.int32, device="cuda")).to(torch.int16).contiguous()   # ~6% density
        grid_dev = torch.full((16,), -1, dtype=torch.int16, device="cuda")
        out_dev = torch.empty((n_lay, 2), dtype=torch.int32, device="cuda")
        for _ in range(3):
            eng.eval_compact_dev(grid_dev.data_ptr(), 16, 16, lay_dev.data_ptr(), n_lay, out_dev.data_ptr())
        ts = []
        for _ in range(10):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.eval_compact_dev(grid_dev.data_ptr(), 16, 16, lay_dev.data_ptr(), n_lay, out_dev.data_ptr())
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ms = float(np.mean(ts))
        gbs = n_lay * (32 + 8) / (ms * 1e-3) / 1e9
        vrate, vthreads, vsample = cpu_validate_rate(grid.data, seconds=5.0)
        line["eval_kernel"] = {"layouts_per_s": n_lay / (ms * 1e-3), "ms": ms, "n": n_lay, "bytes_per_layout": 40,
                               "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "peak_source": hbm_src},
                               "int_gops": 19 * 16 * n_lay / (ms * 1e-3) / 1e9, "int_note": "A_eval = 19 ops x 16 row words per layout (SURVEY.md §8d accounting)",
                               "cpu_validate_layouts_per_s": vrate, "cpu_validate_cores": vthreads, "cpu_validate_sample": vsample}
        # ---------------- kernel (c): CNF check of 131072 witness assignments against the encoder's clauses (incl. the totalizer
        # of the at-most-15 bound): the SLS witness, completed by unit propagation, replicated; every 64th copy has one
        # support removed (those must come back falsified)
        enc = T.Encoding.encode(T.PLATFORMS_DEFAULT[:1], grid)
        cnf = enc.with_limits(T.PlatformLimits.new_unweighted({T.PlatformDef(1, 1): 15}))
        dev = eng.upload_cnf(cnf)
        res, wit = eng.solve_upper_bound(grid, card_limit=OPTIMUM_RECT16, seed=300)
        full = np.full((1, cnf.n_vars + 1), 2, np.uint8)
        base_a = eng.layout_to_assignment(enc, wit)
        full[0, : len(base_a)] = base_a
        prop, conflict, rounds = dev.propagate(full)
        prop[prop == 2] = 0
        assert conflict[0] < 0 and dev.check(prop)[0][0] == 0
        a = np.repeat(prop, 131072, axis=0)     # 4096 words per variable and polarity: long enough a launch to time the kernel, not its launch
        first_support = int(enc.vars().plat_var[[p.y * 16 + p.x for p in wit.platforms().values()][0], 0])
        a[::64, first_support] = 0
        nf, _ = dev.check(a)
        nf, _ = dev.check(a)
        assert (nf[::64] > 0).all() and nf.reshape(-1, 64)[:, 1:].sum() == 0
        cnf_ms = eng.stats()["device_ms"]
        nbw = (len(a) + 31) // 32
        cnf_bytes = 2 * (cnf.n_vars + 1) * nbw * 4 + 8 * len(a)      # both bit-sliced planes read once + (count, first) per assignment written
        cnf_ops = len(cnf.lits) * nbw                                # one logic op per literal per 32 assignments (DESIGN.md A_cnf): thread-ops
        cnf_reads = len(cnf.lits) * nbw * 4                          # ... and one 4-byte plane word per literal and word (L2 traffic: a variable occurs in ~3 clauses)
        line["cnf_kernel"] = {"clause_evals_per_s": cnf.n_clauses * len(a) / (cnf_ms * 1e-3), "clauses": cnf.n_clauses, "ms": cnf_ms,
                              "roofline": {"bound": "hbm", "achieved": cnf_bytes / (cnf_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                           "frac": cnf_bytes / (cnf_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                                           "plane_reads_gbs": cnf_reads / (cnf_ms * 1e-3) / 1e9, "int_gops": cnf_ops / (cnf_ms * 1e-3) / 1e9,
                                           "note": "algorithmic bytes = both bit-sliced assignment planes once + results"},
                              "literals": int(len(cnf.lits)), "assignments": len(a), "propagation_rounds": rounds,
                              "input": "SLS witness completed by unit propagation x 131072, every 64th with one support removed"}
        # ---------------- the REPL flow end to end (BASELINE.json configs[0] and [2]): `load test/exN.toml; solve`
        line["repl_loop"] = {"gpu_seeded": repl_loop_gpu(eng, REPL_INSTANCES), "cpp_driver": repl_loop_cpp_driver(REPL_INSTANCES), "cpu": repl_loop_cpu(REPL_INSTANCES),
                             "note": "crates/repl/src/main.rs:280-366 end to end = time to the PROVEN optimum, wall ms: the loop with the GPU engine answering the SAT iterations, its "
                                     "certified lower bounds closing the gap where they can (exact_solves = 0) and the exact solver (oracle CDCL standing in for Glucose, as on the CPU side) "
                                     "called only for what is left, against the same loop on the CPU alone (1 solver thread); cpp_driver = the same loop in C++ over the C ABI (the Rust shim's call "
                                     "sequence; the certified bounds answer UNSAT inside tss_solve_instance), warm median of 21 solves in one process"}
        # ---------------- single-solve latencies of the other named instances through the C ABI
        fx = json.load(open(os.path.join(ROOT, "tests", "golden", "fixtures.json")))
        ex1_rows = fx["ex1"]["grid"]   # test/ex1.toml
        ex1 = T.WorldGrid.from_toml("[world]\ngrid = [\n" + "".join(f'    "{r}",\n' for r in ex1_rows) + "]\n")
        t1s = []
        for i in range(7):
            t0 = time.perf_counter()
            res, lay3 = eng.solve_upper_bound(ex1, T.PLATFORMS_DEFAULT, card_limit=1, seed=1 + i)
            t1s.append((time.perf_counter() - t0) * 1e3)
            assert res == T.SAT and lay3.platform_count() == 1
        line["other_configs"]["c1"] = {"workload": "test/ex1.toml with the REPL's default-8 platform set (BASELINE.json configs[0])", "count": lay3.platform_count(),
                                       "proven_optimum": proven_optimum("ex1/default8"), "ms": float(np.median(t1s[2:])),
                                       "note": "tss_solve_upper_bound(card_limit=1) from host buffers, median of 5 calls after 2 warm-up calls"}
        ex2 = np.array([[1 if (i < len(r) and r[i] == "X") else 0 for i in range(max(len(q) for q in fx["ex2"]["grid"]))] for r in fx["ex2"]["grid"]], np.uint8)
        ex2[8:10, 8:10] = 1          # README terrain = test/ex2.toml with (8,8),(9,8),(8,9),(9,9) set to ceiling (SURVEY.md §8d)
        opt3 = proven_optimum("readme/1x1")
        t3s = []
        for i in range(7):
            t0 = time.perf_counter()
            res, lay2 = eng.solve_upper_bound(T.WorldGrid(ex2), card_limit=opt3, seed=40 + i)
            t3s.append((time.perf_counter() - t0) * 1e3)
            assert res == T.SAT and lay2.platform_count() == opt3
        line["other_configs"]["c3"] = {"workload": "README 21x16 terrain, 1x1 supports (BASELINE.json configs[2])", "count": opt3, "proven_optimum": opt3, "ms": float(np.median(t3s[2:])),
                                       "note": "tss_solve_upper_bound(card_limit=14) from host buffers, median of 5 calls after 2 warm-up calls; the README transcript stops at 15 (README.md:117-119)"}
        # ---------------- the placement search (platform sets beyond {1x1}: what the REPL actually runs, main.rs:254) in throughput mode
        sp = eng.search(T.WorldGrid(named_grid(fx, "ex2")), T.PLATFORMS_DEFAULT, seed=1, n_chains=info["sm_count"] * 32)
        for _ in range(2):
            sp.run(512, 0)
        sp.best_count()
        p0 = eng.stats()
        pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pa.record()
        for _ in range(5):
            sp.run(2048, 0)
        pb.record()
        torch.cuda.synchronize()
        pbest = sp.best_count()
        p1 = eng.stats()
        pms = pa.elapsed_time(pb)
        line["other_configs"]["placement_search"] = {
            "workload": "test/ex2.toml, the REPL's default-8 platform set, sls_multi_kernel (one chain per warp, objective = number of platforms)",
            "flips_per_s": (p1["sls_flips"] - p0["sls_flips"]) / (pms * 1e-3), "placements_scored_per_s": (p1["candidates_scored"] - p0["candidates_scored"]) / (pms * 1e-3),
            "sls_steps_per_s": (p1["sls_steps"] - p0["sls_steps"]) / (pms * 1e-3), "chains": sp.n_chains, "ms": pms, "best_count": pbest,
            "proven_optimum": proven_optimum("ex2/default8")}
        sp.close()
        # ---------------- CPU baseline (bounded sample, rank 0, N = 1): the same step rule, chains and unit on the host cores
        rate, epoch_ms, threads, n_cpu, cpu_best, sample = cpu_flips(grid.data, args.epoch_steps, 3, 12)
        given, unbounded = cdcl_time_to_optimum(grid.data, OPTIMUM_RECT16)      # 1 thread like the reference
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                                "time_to_optimal": {"given_bound_ms": given, "from_unbounded_ms": unbounded,
                                                    "note": "oracle CDCL (Glucose stand-in, crates/repl/src/main.rs:280-366), 1 solver thread as in the reference (solver_runner.rs:15); "
                                                            "the UNSAT proof of 14 (minutes, tests/golden/proofs.json) is not included"}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
