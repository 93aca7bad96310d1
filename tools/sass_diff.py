#!/usr/bin/env python
"""SASS of every kernel in two builds of libfairmarl.so, compared function by function (cuobjdump -sass, instruction
text line by line; kernels keyed by demangled name).  usage: sass_diff.py OLD.so NEW.so > profiles/..."""
import hashlib
import re
import subprocess
import sys


def kernels(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(.*?);", line)
        if m and name:
            funcs[name].append(m.group(1).strip())
    names = subprocess.run(["c++filt"], input="\n".join(funcs), capture_output=True, text=True).stdout.splitlines()
    return {nice: funcs[mangled] for mangled, nice in zip(funcs, names)}


old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
# a kernel that gained a trailing defaulted template parameter keeps its parent's name for the default value
new = {(k2 if k not in old and (k2 := k.replace(", false>(", ">(", 1)) in old else k): v for k, v in new.items()}
print("SASS of every kernel in libfairmarl.so: parent commit vs this change (cuobjdump -sass, instruction text compared "
      "line by line; kernels keyed by demangled name)\n")
same = diff = 0
for k in sorted(old):
    if k not in new:
        continue
    a, b = old[k], new[k]
    eq = a == b
    same += eq
    diff += not eq
    print(f"{'identical' if eq else 'DIFFERENT':10} {len(a):6} / {len(b):6} instr  sha1 "
          f"{hashlib.sha1(chr(10).join(b).encode()).hexdigest()[:12]}  {k[:110]}")
added, removed = sorted(set(new) - set(old)), sorted(set(old) - set(new))
for k in added:
    print(f"{'new':10} {'':6}   {len(new[k]):6} instr  {k[:120]}")
for k in removed:
    print(f"{'removed':10} {len(old[k]):6}            {k[:120]}")
print(f"\n{same} kernels identical, {diff} different, {len(added)} new, {len(removed)} removed")
