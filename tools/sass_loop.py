#!/usr/bin/env python
"""Print the instruction mix of the innermost (hottest) loop of each kernel in a cubin / .so / executable.

Usage: sass_loop.py <binary> [kernel-substring] [loops per kernel]
       sass_loop.py --compare <binary A> <binary B>
A loop is a backward branch; for every kernel the loop with the most instructions is reported.
Used to check instruction budgets per cell before spending GPU time (see DESIGN.md, "Instruction budget").

--compare lists the kernels only in A, only in B, and those whose instructions differ, and exits non-zero if there is
any: a refactor that leaves every kernel's SASS as it was cannot change what a kernel computes or how fast it runs.  The hash nvcc gives
each file's anonymous namespace differs from build to build and is left out of the names.
"""
import re, subprocess, sys, collections

def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    name, body = None, []
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            if name: yield name, body
            name, body = m.group(1), []
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m and name:
            body.append((int(m.group(1), 16), m.group(2).strip()))
    if name: yield name, body

def loops(body):
    res = []
    for idx, (addr, ins) in enumerate(body):
        m = re.search(r"\bBRA(?:\.\w+)*\s+(?:\S+,\s*)?(0x[0-9a-f]+)", ins)
        if m:
            tgt = int(m.group(1), 16)
            if tgt <= addr:
                res.append([i for a, i in body if tgt <= a <= addr])
    return res

def normalised(path):
    res = {}
    for name, body in kernels(path):
        name = re.sub(r"_GLOBAL__N__[0-9a-f]+_(\d+_\w+?)_[0-9a-f]{8}", r"_GLOBAL__N__\1", name)
        res.setdefault(name, []).append([ins for _, ins in body])
    return res

def compare(path_a, path_b):
    a, b = normalised(path_a), normalised(path_b)
    only_a, only_b = sorted(a.keys() - b.keys()), sorted(b.keys() - a.keys())
    differ = sorted(n for n in a.keys() & b.keys() if a[n] != b[n])
    for title, names in ((f"only in {path_a}", only_a), (f"only in {path_b}", only_b), ("instructions differ", differ)):
        print(f"{title}: {len(names)}")
        for n in names: print(f"  {n}")
    print(f"identical: {len(a.keys() & b.keys()) - len(differ)} kernels")
    return 1 if only_a or only_b or differ else 0

def main():
    if sys.argv[1] == "--compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    path = sys.argv[1]; sub = sys.argv[2] if len(sys.argv) > 2 else ""
    for name, body in kernels(path):
        if sub not in name: continue
        ls = loops(body)
        if not ls:
            print(f"{name}: no loop ({len(body)} instrs)"); continue
        for l in sorted(ls, key=len, reverse=True)[:int(sys.argv[3]) if len(sys.argv) > 3 else 1]:
            c = collections.Counter(re.sub(r"^@!?U?P\d+\s+", "", i).split()[0].split(".")[0] for i in l)
            print(f"{name}: loop {len(l)} instrs: " + " ".join(f"{k}={v}" for k, v in c.most_common()))

if __name__ == "__main__":
    main()
