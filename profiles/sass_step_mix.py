"""Static SASS mix of the step loop of the thread-per-chain SLS kernels (no GPU needed): the stand-in for a per-line
profile when none can be taken.  Compiles csrc/sls_t16.cu and csrc/sls_p16.cu with the library's flags, disassembles them
with line info and counts the instructions attributed to each part of a chain step (as source line ranges):

    python profiles/sass_step_mix.py [OUTDIR]

`flip` is inlined three times (list start-up, removal, addition) and reported per copy; the addition block is one copy
per step.  The removal scan is reported per support scored: t16's loop is unrolled by 4 (plus a remainder copy), so its
instructions are divided by 5; p16 scans its CAP cached slots fully unrolled, divided by CAP (the loop over list entries
past CAP, which only dense warm starts reach, is not counted).  The scan counts every instruction between its first and
last one, the inlined helpers (anchor, byte packs, the loss) included; elsewhere instructions attributed to small helpers
defined outside the ranges (pick_rotated, the byte-pack functions) are not counted, so the figures compare parts of the
two kernels, not whole steps."""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from timberborn_support_solver_b200 import build as B  # noqa: E402

CUDA = os.path.dirname(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")))
FLAGS = [f for f in B.NVCC_FLAGS if f not in ("-shared", "-cudart", "static", "-ldl")]


def ranges(src):
    """source line ranges of the parts of a step, found by the code's own landmarks"""
    lines = open(src).read().split("\n")
    find = lambda pat, start=0: next(i + 1 for i in range(start, len(lines)) if re.search(pat, lines[i]))
    flip = find(r"__device__ __forceinline__ void flip\(")
    shl = find(r"uint32_t shl_clamped\(")
    add_key = find(r"^template <int DX, int DY>")
    kern = find(r"^__global__ void")
    cap = re.search(r"constexpr int CAP = (\d+);", "\n".join(lines))
    if cap:     # p16: the unrolled scan of the cached slots, up to the overflow loop
        rm0 = find(r"for \(int i = 0; i < CAP; i\+\+\) \{", find(r"const int kw = ", kern))
        rm1, rm_part = find(r"if \(kw > CAP\)", rm0), f"removal, per cached support (scan / {cap.group(1)})"
    else:
        rm0 = find(r"for \(int i = 0; i < k; i\+\+, mult", kern)
        rm1, rm_part = find(r"const int best_i = ", rm0), "removal, per support (scan / 5)"
    ad0 = find(r"const int y = pick_rotated\(", rm1)
    ad1 = find(r"flip<true>\(sm, tid, v, ", ad0)
    return {"flip (per copy)": (flip, shl, 3, False), rm_part: (rm0, rm1, int(cap.group(1)) if cap else 5, True),
            "addition: 25 candidates (add_key/add_column)": (add_key, kern, 1, False), "addition: fetch, pick, tabu window, decode": (ad0, ad1, 1, False)}


def mix(name, out):
    src = os.path.join(B.CSRC, name + ".cu")
    obj = os.path.join(out, name + ".o")
    ptx = subprocess.run([os.path.join(CUDA, "bin", "nvcc"), *FLAGS, "-Xptxas", "-v", "-c", src, "-o", obj], cwd=B.CSRC, capture_output=True, text=True, check=True).stderr
    regs = re.findall(r"_kernel.*\n.*\n.*?(\d+) bytes spill stores.*\n.*?Used (\d+) registers", ptx)
    subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-xelf", "all", obj], cwd=out, check=True, capture_output=True)
    cubin = next(os.path.join(out, f) for f in os.listdir(out) if f.startswith(name) and f.endswith(".cubin"))
    sass = subprocess.run([os.path.join(CUDA, "bin", "nvdisasm"), "-g", "-c", cubin], capture_output=True, text=True, check=True).stdout
    rng = ranges(src)
    per = collections.defaultdict(collections.Counter)
    ins = []   # (our source line or None, opcode) in address order
    line, ours = 0, False
    for l in sass.split("\n"):
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            ours, line = m.group(1).endswith(name + ".cu"), int(m.group(2))
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)", l)
        if m:
            ins.append((line if ours else None, m.group(1)))
    for part, (a, b, _, span) in rng.items():
        hit = [j for j, (ln, _) in enumerate(ins) if ln is not None and a <= ln < b]
        for j in range(hit[0], hit[-1] + 1) if span else hit:
            per[part][ins[j][1]] += 1
    print(f"{name}: {regs[0][1] if regs else '?'} registers, {regs[0][0] if regs else '?'} bytes spilled")
    for part, (a, b, div, _) in rng.items():
        c = per[part]
        top = ", ".join(f"{op} {n / div:.1f}" for op, n in c.most_common(8))
        print(f"  {part:48s} {sum(c.values()) / div:6.1f}   ({top})")


if __name__ == "__main__":
    with tempfile.TemporaryDirectory() as tmp:
        out = sys.argv[1] if len(sys.argv) > 1 else tmp
        for k in ("sls_t16", "sls_p16"):
            mix(k, out)
