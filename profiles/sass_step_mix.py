"""Static SASS mix of the step loop of the thread-per-chain SLS kernels (no GPU needed): the stand-in for a per-line
profile when none can be taken.  Compiles csrc/sls_t16.cu and csrc/sls_p16.cu with the library's flags, disassembles them
with line info and counts the instructions attributed to each part of a chain step (as source line ranges in the kernel's
file, in sls_thread.cuh, which holds the step both kernels share, and in sls_spec.hpp; an instruction counts at its
innermost inlined frame, except that the load / store accessors and the plane and key helpers of sls_thread.cuh count
where they are called):

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
# opcodes issued to the integer-ALU pipe (the "ALU" column): the pipe that bounds both kernels, one warp instruction every
# 2 clocks per scheduler (DESIGN.md).  IMAD, POPC and the memory instructions issue elsewhere.
ALU = {"LOP3", "SHF", "PRMT", "ISETP", "SEL", "VIMNMX", "VIADDMNMX", "IADD3", "LEA", "R2P", "PLOP3"}


def read(path):
    return open(path).read().split("\n")


def find(lines, pat, start=0):
    return next(i + 1 for i in range(start, len(lines)) if re.search(pat, lines[i]))


def body(lines, pat, start=0):
    """[first, last + 1) source lines of the function whose signature matches pat (braces matched from its first line)"""
    a = find(lines, pat, start)
    depth, opened = 0, False
    for i in range(a - 1, len(lines)):
        depth += lines[i].count("{") - lines[i].count("}")
        opened = opened or "{" in lines[i]
        if opened and depth == 0:
            return a, i + 2


def ranges(name):
    """source line ranges of the parts of a step, found by the code's own landmarks: {part: ([(file, first, end)], divisor, span)}.
    The kernel's own file holds its representation, sls_thread.cuh the shared step and sls_spec.hpp the diamond decoding."""
    src, hdr, spec = (os.path.join(B.CSRC, f) for f in (name + ".cu", "sls_thread.cuh", "sls_spec.hpp"))
    L, H, S = read(src), read(hdr), read(spec)
    cap = re.search(r"constexpr int CAP = (\d+);", "\n".join(L))
    if cap:     # p16: the unrolled scan of the cached slots, up to the overflow loop
        rm0 = find(L, r"for \(int i = 0; i < CAP; i\+\+\) \{", find(L, r"const int kw = "))
        rm1, rm_part = find(L, r"if \(kw > CAP\)", rm0), f"removal, per cached support (scan / {cap.group(1)})"
    else:
        rm0 = find(L, r"for \(int i = 0; i < k; i\+\+, mult")
        rm1, rm_part = find(L, r"const int best_i = ", rm0), "removal, per support (scan / 5)"
    add0 = find(L, r"__device__ __forceinline__ void add\(")
    run = find(H, r"void run_chains\(")
    return {"flip (per copy)": ([(src, *body(L, r"__device__ __forceinline__ void flip\("))], 3, False),
            rm_part: ([(src, rm0, rm1)], int(cap.group(1)) if cap else 5, True),
            "addition: 25 candidates (add_key/add_column)": ([(hdr, *body(H, r"uint32_t add_key\(")), (hdr, *body(H, r"uint32_t add_column\(")),
                                                              (src, *body(L, r"void slab\(")), (src, *body(L, r"uint32_t gain\("))], 1, False),
            "addition: fetch, pick, tabu window, decode": ([(src, *body(L, r"Nbhd fetch\(")), (src, add0, find(L, r"flip<true>\(sm, tid, v, ", add0)),
                                                            (hdr, find(H, r"const auto N = R\.fetch\(", run), find(H, r"const int v = add_site\(", run) + 1),
                                                            (hdr, *body(H, r"int add_site\(")), (spec, *body(S, r"void diamond_cell\("))], 1, False)}


def transparent(name):
    """sls_thread.cuh functions whose instructions count where they are called: the checked loads / stores (the macros of
    earlier kernels) and the key and plane helpers that used to be written out at their call sites"""
    hdr = os.path.join(B.CSRC, "sls_thread.cuh")
    H = read(hdr)
    return [(hdr, *body(H, pat)) for pat in (r" T ld\(", r"uint2 ld_tab\(", r"uint32_t& st\(", r"uint32_t flip_word\(", r"uint32_t remove_key\(")]


def mix(name, out):
    src = os.path.join(B.CSRC, name + ".cu")
    obj = os.path.join(out, name + ".o")
    ptx = subprocess.run([os.path.join(CUDA, "bin", "nvcc"), *FLAGS, "-Xptxas", "-v", "-c", src, "-o", obj], cwd=B.CSRC, capture_output=True, text=True, check=True).stderr
    regs = re.findall(r"_kernel.*\n.*\n.*?(\d+) bytes spill stores.*\n.*?Used (\d+) registers", ptx)
    subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-xelf", "all", obj], cwd=out, check=True, capture_output=True)
    cubin = next(os.path.join(out, f) for f in os.listdir(out) if f.startswith(name) and f.endswith(".cubin"))
    sass = subprocess.run([os.path.join(CUDA, "bin", "nvdisasm"), "-gi", "-c", cubin], capture_output=True, text=True, check=True).stdout
    rng, skip = ranges(name), transparent(name)
    inside = lambda f, ln, spans: any(f == g and a <= ln < b for g, a, b in spans)
    per = collections.defaultdict(collections.Counter)
    ins = []   # (source file and line the instruction counts at, opcode) in address order
    chain, fresh = [], False   # the instruction's inlining chain, innermost frame first
    for l in sass.split("\n"):
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            chain, fresh = ([] if not fresh else chain) + [(os.path.realpath(m.group(1)), int(m.group(2)))], True
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)", l)
        if m:
            fresh = False
            at = next(((f, ln) for f, ln in chain if not inside(f, ln, skip)), (None, 0))
            ins.append((at, m.group(1)))
    for part, (spans, _, span) in rng.items():
        hit = [j for j, (at, _) in enumerate(ins) if inside(*at, spans)]
        for j in range(hit[0], hit[-1] + 1) if span else hit:
            per[part][ins[j][1]] += 1
    print(f"{name}: {regs[0][1] if regs else '?'} registers, {regs[0][0] if regs else '?'} bytes spilled")
    print(f"  {'':48s} {'all':>6s} {'ALU':>6s}")
    for part, (_, div, _) in rng.items():
        c = per[part]
        alu = sum(n for op, n in c.items() if op in ALU)
        top = ", ".join(f"{op} {n / div:.1f}" for op, n in c.most_common(8))
        print(f"  {part:48s} {sum(c.values()) / div:6.1f} {alu / div:6.1f}   ({top})")


if __name__ == "__main__":
    with tempfile.TemporaryDirectory() as tmp:
        out = sys.argv[1] if len(sys.argv) > 1 else tmp
        for k in ("sls_t16", "sls_p16"):
            mix(k, out)
