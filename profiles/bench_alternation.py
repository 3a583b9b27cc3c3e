"""`bench.py --gpus 1 --quick` alternated between builds of libtss in one run, so that every build sees the same card, clocks
and neighbours, and the spread between rounds shows the noise; then `--dump-outputs` of every build compared byte for byte
with the first one's.

    python profiles/bench_alternation.py OUTDIR [--rounds N] [--bench-args "..."] LABEL=LIB [LABEL=LIB ...]

LIB is the path of a libtss build (loaded through TSS_LIB), or "tree" for the library built in this tree.  Prints the
card's name, power limit and max SM clock, one line per run, the min-max per build and whether each build's dump is
byte-identical to the first build's, and writes every bench line to OUTDIR/alternation.jsonl."""
import argparse
import json
import os
import shlex
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("builds", nargs="+", metavar="LABEL=LIB")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--bench-args", default="", help="extra bench.py arguments (e.g. --kernel 3)")
    a = ap.parse_args()
    builds = [b.split("=", 1) for b in a.builds]
    os.makedirs(a.out, exist_ok=True)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    print(f"# bench.py --gpus 1 --quick {a.bench_args} alternated in one run: " + ", ".join(f"{l} = {p}" for l, p in builds))
    print("name, power.limit, clocks.max.sm:", smi.strip().split("\n")[0])
    rates = {l: [] for l, _ in builds}

    def bench(label, lib, extra):
        env = dict(os.environ)
        env.pop("TSS_LIB", None)
        if lib != "tree":
            env["TSS_LIB"] = os.path.abspath(lib)
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--quick", *shlex.split(a.bench_args), *extra]
        r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
        lines = [l for l in r.stdout.split("\n") if l.startswith("{")]
        if r.returncode or not lines:
            print(f"{label:10s} FAILED rc {r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}", flush=True)
            sys.exit(1)
        return json.loads(lines[-1])

    with open(os.path.join(a.out, "alternation.jsonl"), "w") as f:
        for r in range(a.rounds):
            for label, lib in (builds if r % 2 == 0 else builds[::-1]):   # a drift within a round does not always meet the same build
                line = bench(label, lib, [])
                rates[label].append(line["value"])
                f.write(json.dumps(dict(line, build=label)) + "\n")
                print(f"{label:10s} value {line['value']:.4e} ms_per_step {line['ms_per_step']:.3f} kernel '{line['run']['kernel']}' "
                      f"chains {line['run']['chains_per_gpu']} best {line['best_count']} clocks {json.dumps(line.get('clocks'))}", flush=True)
    base = builds[0][0]
    for label, _ in builds:
        lo, hi = min(rates[label]), max(rates[label])
        print(f"{label:10s} {lo / 1e9:.2f}-{hi / 1e9:.2f} G flips/s, x{lo / max(rates[base]):.4f}-{hi / min(rates[base]):.4f} against {base}")
    dumps = {}
    with tempfile.TemporaryDirectory() as tmp:   # up to 64 MB per build: compared here, not kept
        for label, lib in builds:
            d = os.path.join(tmp, "dump_" + label)
            bench(label, lib, ["--dump-outputs", d])
            dumps[label] = {n: open(os.path.join(d, n), "rb").read() for n in sorted(os.listdir(d))}
    for label, _ in builds[1:]:
        same = dumps[label].keys() == dumps[base].keys() and all(dumps[label][n] == dumps[base][n] for n in dumps[base])
        print(f"dump {label} vs {base}: {len(dumps[label])} files, byte-identical: {same}")


if __name__ == "__main__":
    main()
