#!/usr/bin/env python
"""Compare two `cuobjdump -sass` dumps of librlsde_b200.so function by function (instruction encodings only: the text
column's width varies with a function's longest line).

    cuobjdump -sass parent/librlsde_b200.so > old.txt; cuobjdump -sass rl_sde_is_b200/librlsde_b200.so > new.txt
    python tools/sass_identity.py old.txt new.txt

A parent function missing from the new dump is looked up with one more template argument `false` (`Lb0E`) appended:
kernels that gained a defaulted trailing bool parameter (BRIDGE) keep their old code under that name."""
import re, sys

def funcs(path):
    out, name, buf = {}, None, []
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name: out[name] = "".join(buf)
            name, buf = m.group(1), []
            continue
        if name is None or not line.lstrip().startswith("/*"):      # instructions and their encodings only
            continue
        buf.append(line)
    if name: out[name] = "".join(buf)
    return out

def enc(body):
    return re.findall(r'/\* (0x[0-9a-f]{16}) \*/', body)


old, new = funcs(sys.argv[1]), funcs(sys.argv[2])
same = changed = removed = 0
used = set()
lines = []
for n, body in old.items():
    m = n
    if m not in new:
        mm = re.match(r"(_ZN5rlsde\d+\w+?I(?:L[^E]+E)+)(E.*)", n)
        if mm and mm.group(1) + "Lb0E" + mm.group(2) in new:
            m = mm.group(1) + "Lb0E" + mm.group(2)
    if m not in new:
        removed += 1; lines.append(f"REMOVED {n}"); continue
    used.add(m)
    if enc(new[m]) == enc(body): same += 1
    else: changed += 1; lines.append(f"CHANGED {n}")
added = [n for n in new if n not in used]
print(f"parent: {len(old)} functions; this change: {len(new)}")
print(f"identical SASS: {same}; changed: {changed}; removed: {removed}; added: {len(added)}")
renamed = sum(1 for n in old if n not in new)
print(f"compared under the name with BRIDGE = false appended: {renamed - removed}")
for l in lines: print(l)
for n in sorted(added):
    print(f"ADDED {n} ({sum(1 for l in new[n].splitlines() if l.lstrip().startswith('/*') and '*/' in l and not l.lstrip().startswith('/* 0x'))} instructions)")
