#!/usr/bin/env python
"""Registers, stack frame, local and shared memory per kernel of the built library, from `cuobjdump -res-usage`.

usage: ptxas_report.py [path/to/libnanorepeat_b200.so]   (default: the in-tree library that `make` builds)

One line per kernel, sorted by name, so that two builds compare with `diff`.  Spills live in the stack frame:
cuobjdump reports no separate spill count (`nvcc -Xptxas -v` does, per translation unit)."""
import os
import re
import subprocess
import sys

here = os.path.dirname(os.path.abspath(__file__))
lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(here, "..", "nanorepeat_b200", "libnanorepeat_b200.so")
out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-res-usage", lib], capture_output=True, text=True, check=True).stdout
rows, name = {}, None
for ln in out.splitlines():
    m = re.match(r"\s*Function (\S+):$", ln)
    if m:
        d = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        d = d.replace("(anonymous namespace)::", "")
        name = re.sub(r"^void ", "", d.split("(")[0])       # drop the parameter list: templates name the variant
        continue
    if name:
        f = dict(re.findall(r"(\w+(?:\[\d+\])?):(\d+)", ln))
        rows[name] = f"regs={f.get('REG')} stack={f.get('STACK')} local={f.get('LOCAL')} shared={f.get('SHARED')}"
        name = None
width = max(map(len, rows), default=0)
for k in sorted(rows):
    print(f"{k:{width}s}  {rows[k]}")
