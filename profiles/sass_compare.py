#!/usr/bin/env python
"""Per-kernel comparison of two builds of one CUDA source: SASS instruction text, opcode histogram and the
`-Xptxas -v` register / spill lines of every kernel the old object has.  A kernel that gained a defaulted template
argument (e.g. `softmax_kl_regs_kernel<F, T, I>` -> `<F, T, I, true>`), or a leading `float` score-type argument
(e.g. `rank_targets_kernel<true>` -> `<float, true>`), is matched to its old name.

    nvcc ... -Xptxas -v -c src.cu -o old.o 2> old.ptxas      (parent commit)
    nvcc ... -Xptxas -v -c src.cu -o new.o 2> new.ptxas      (this change)
    python profiles/sass_compare.py old.o old.ptxas new.o new.ptxas
"""
import collections
import re
import subprocess
import sys


def demangle(n):
    return subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip().split("(")[0]


def sass(obj):
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    k, fn = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1); k[fn] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and fn:
            k[fn].append(m.group(1).strip())
    return k


def ptxas(path):
    d, fn = {}, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(\S+)'", line) or re.search(r"Function properties for (\S+)", line)
        if m:
            fn = m.group(1)
        if fn and ("registers" in line or "spill" in line):
            d.setdefault(fn, []).append(line.strip().split("info    : ")[-1])
    return d


old_o, old_p, new_o, new_p = sys.argv[1:5]
a, b, pa, pb = sass(old_o), sass(new_o), ptxas(old_p), ptxas(new_p)
new_by_old = {}
for n in b:
    d = demangle(n)
    new_by_old[d] = n
    new_by_old.setdefault(re.sub(r", true>$", ">", d), n)
    new_by_old.setdefault(re.sub(r"<float, ", "<", d), n)
same = 0
for n in sorted(a, key=demangle):
    d = demangle(n)
    m = new_by_old.get(d)
    if m is None:
        print(f"MISSING {d}")
        continue
    ok_text, ok_regs = a[n] == b[m], pa.get(n) == pb.get(m)
    ok_hist = collections.Counter(i.split()[0] for i in a[n]) == collections.Counter(i.split()[0] for i in b[m])
    same += ok_text and ok_regs and ok_hist
    print(f"{'SAME' if ok_text and ok_regs and ok_hist else 'DIFF'} text={ok_text} histogram={ok_hist} regs={ok_regs} "
          f"{d}{'' if m == n else ' (now ' + demangle(m) + ')'}: {len(a[n])} instructions; {' | '.join(pb.get(m, []))}")
matched = {new_by_old.get(demangle(n)) for n in a}
for n in sorted(set(b) - matched, key=demangle):
    print(f"NEW {demangle(n)}: {len(b[n])} instructions; {' | '.join(pb.get(n, []))}")
print(f"# {same} of {len(a)} existing kernels unchanged")
