#!/usr/bin/env python
"""Compares the machine code of two builds of libgfr_b200.so (no GPU needed): the SASS of every kernel, with addresses
and encodings stripped, and `cuobjdump -res-usage` (registers, stack, shared / local memory) per kernel.  For each
kernel whose SASS differs it prints the differing lines and whether the two instruction lists hold the same
instructions in another order.  usage: python profiles/sass_compare.py OLD.so NEW.so"""
import collections
import difflib
import re
import subprocess
import sys

ANON = re.compile(r"_GLOBAL__N__[0-9a-f]{8}_\d+_gfr_b200_cu_[0-9a-f]{8}")   # anonymous namespace: its hash depends on the source text


def short(name):
    m = re.search(r"\d+([a-z_]+_kernel)(I.*?E)?E", name)
    if not m:
        return name[:60]
    return m.group(1) + ("<" + ",".join(re.findall(r"L[ib](\d+)E", m.group(2))) + ">" if m.group(2) else "")


def sass(lib):
    text = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = ANON.sub("_GLOBAL__N_", m.group(1))
            out[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(.*?)\s*;", line)
        if m and cur:
            out[cur].append(ANON.sub("_GLOBAL__N_", m.group(1)))
    return out


def resources(lib):
    text = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            cur = ANON.sub("_GLOBAL__N_", m.group(1))
        elif cur and "REG:" in line:
            out[cur] = " ".join(line.split()[:4])
            cur = None
    return out


def main():
    old, new = sys.argv[1], sys.argv[2]
    a, b = sass(old), sass(new)
    ra, rb = resources(old), resources(new)
    print(f"# kernels: {len(a)} / {len(b)}, same names: {set(a) == set(b)}; "
          f"instructions: {sum(map(len, a.values()))} / {sum(map(len, b.values()))}")
    differ = [f for f in sorted(a) if a[f] != b.get(f)]
    print(f"# kernels with different SASS: {len(differ)}; with different resource usage: "
          f"{sum(ra[f] != rb.get(f) for f in ra)}")
    for f in differ:
        same = collections.Counter(a[f]) == collections.Counter(b.get(f, []))
        print(f"\n{short(f)}: {len(a[f])} / {len(b.get(f, []))} instructions, same instructions reordered: {same}")
        for line in difflib.unified_diff(a[f], b.get(f, []), lineterm="", n=3):
            if not line.startswith(("---", "+++")):
                print("   ", line)
    print("\n# resource usage per kernel (old | new)")
    for f in sorted(ra, key=short):
        print(f"{short(f):36s} {ra[f]:44s} | {rb.get(f)}")


if __name__ == "__main__":
    main()
