"""Per-kernel SASS identity of two builds of one source file: `cuobjdump -sass` of each cubin with /*addr*/ and /* 0x... */
encoding comments stripped (branch targets and constant-bank offsets kept), compared kernel by kernel; registers and spills
from the two `-Xptxas -v` reports.  A kernel that gained a `false` template argument is matched to its old name.

    nvcc <build.NVCC_FLAGS without -shared -cudart static -ldl> -cubin -Xptxas -v -o old.cubin old.cu 2> old.txt   (same for new)
    python profiles/sass_identity.py old.cubin old.txt new.cubin new.txt
"""
import re, subprocess, sys

def sass(cubin):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); funcs[cur] = []; continue
        if cur and re.search(r"/\*[0-9a-f]{4,}\*/", line):
            ins = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)
            ins = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", ins).strip().rstrip(";").strip()
            funcs[cur].append(ins)
    return funcs

def regs(log):
    r, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m: cur = m.group(1)
        m = re.search(r"Used (\d+) registers", line)
        if m and cur: r.setdefault(cur, {})["regs"] = int(m.group(1))
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur: r.setdefault(cur, {})["spill"] = (int(m.group(1)), int(m.group(2)))
    return r

def demangle(n):
    return subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip().split("(")[0]

old, new = sass(sys.argv[1]), sass(sys.argv[3])
ro, rn = regs(sys.argv[2]), regs(sys.argv[4])
mapping = {}
for n in new:
    d = demangle(n)
    cand = [o for o in old if demangle(o).replace(">", ", false>") == d or demangle(o) == d]
    mapping[n] = cand[0] if cand else None
for n, o in mapping.items():
    d = demangle(n)
    if o is None:
        print(f"new        {len(new[n])} instructions, registers {rn.get(n, {}).get('regs')}, spills {rn.get(n, {}).get('spill')}  {d}")
    else:
        same = old[o] == new[n]
        print(f"{'identical' if same else 'DIFFERENT'}  {len(old[o])} / {len(new[n])} instructions, registers {ro.get(o, {}).get('regs')} / {rn.get(n, {}).get('regs')}  {demangle(o)}  ->  {d}")
