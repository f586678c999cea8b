#!/usr/bin/env python
"""STATIC SASS instructions of k_tile_merge per phase (the '// ---- X:' markers of csrc/tile.cuh), from the line info that the
Makefile's -lineinfo puts into libdsa.so.  Static: each instruction of the code counts once, whatever a loop or a branch does
with it at run time (executed counts need a profiler).
usage: python profiles/sass_phases.py [path/to/libdsa.so]   (default: the library of this tree; csrc/tile.cuh next to it)"""
import os
import re
import subprocess
import sys
import tempfile
from collections import Counter

root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else os.path.join(root, "dynamicsparsearrays.jl_b200", "libdsa.so"))
lines = open(os.path.join(os.path.dirname(so), "csrc", "tile.cuh")).read().splitlines()
marks = [(i + 1, l.strip()[8:30]) for i, l in enumerate(lines) if l.strip().startswith("// ---- ")]
kstart = next(i + 1 for i, l in enumerate(lines) if "k_tile_merge(TileArgs" in l)
cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def phase(f, n):
    if f != "tile.cuh":
        return f
    if n < kstart:
        return "helpers (tile_find, ranks)"
    p = "prologue"
    for ln, name in marks:
        if n >= ln:
            p = name
    return p


with tempfile.TemporaryDirectory() as tmp:
    subprocess.check_call([f"{cuda}/bin/cuobjdump", "-xelf", "all", so], cwd=tmp, stdout=subprocess.DEVNULL)
    cubin = next(os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin"))
    sass = subprocess.check_output([f"{cuda}/bin/nvdisasm", "-g", "-c", cubin], text=True)

counts, fn, loc = {}, None, None
for ln in sass.splitlines():
    m = re.match(r"\s*\.text\.(\S*k_tile_merge\S*):", ln)
    if m:
        fn = m.group(1)
        counts[fn] = Counter()
        continue
    if ln.startswith("//---------------------") and "k_tile_merge" not in ln:
        fn = None
    m = re.search(r'//## File "([^"]+)", line (\d+)', ln)
    if m:
        loc = (os.path.basename(m.group(1)), int(m.group(2)))
    elif fn and loc and re.match(r"\s+/\*[0-9a-f]{4,}\*/", ln):
        counts[fn][phase(*loc)] += 1
for fn in sorted(counts):
    c = counts[fn]
    print(f"{fn}: {sum(c.values())} static SASS instructions")
    for k, v in sorted(c.items(), key=lambda kv: -kv[1]):
        print(f"  {v:5d}  {k}")
