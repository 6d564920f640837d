#!/usr/bin/env python
"""Compare the SASS of every nlm_tiled_kernel instantiation in two object files function by function (the trailing
DH template flag is ignored in the key, so objects from before / after that parameter was added line up).
Usage: sass_funcs.py old.o new.o   -- prints IDENTICAL / differs per instantiation.  Used to make sure a change to
nlm_tiled.cuh leaves the instruction schedules of the shipped instantiations untouched (DESIGN.md 4.1 / 4.2a).
Other kernels are keyed on their full name, except the change-detection kernels, which are keyed on kernel and
accumulator so the dual-pol instantiations (`<Acc<T>>`, formerly `<T>`) line up (DESIGN.md 12)."""
import sys, re, subprocess, hashlib
def funcs(path):
    txt = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True).stdout
    out = {}; cur = None
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1); out[cur] = []; continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m and cur is not None:
            out[cur].append(m.group(2).strip())
    return out
def key(name):
    m = re.match(r"_ZN5ndchg\d+(\w+?_kernel)I(?:NS_3AccI(\w)EEE|(\w)E)E", name)
    if m: return "ndchg::%s<Acc<%s>>" % (m.group(1), m.group(2) or m.group(3))
    # template args of nlm_tiled_kernel: strip trailing DH flag if present -> comparable key
    m = re.search(r"nlm_tiled_kernelI(\w)((?:L[ib]\d+E)+)E", name)
    if not m: return name
    args = re.findall(r"L[ib](\d+)E", m.group(2))
    return m.group(1) + "," + ",".join(args[:9])
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
ka = {key(n): n for n in a}; kb = {key(n): n for n in b}
for k in sorted(ka):
    if k not in kb: print(k, "missing in new"); continue
    ia, ib = a[ka[k]], b[kb[k]]
    same = ia == ib
    print("%-40s %6d %6d %s" % (k, len(ia), len(ib), "IDENTICAL" if same else "differs"))
