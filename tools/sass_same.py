"""Kernels that two objects (or libraries) both contain, by mangled name, and whether their cuobjdump -sass text is the same
once instruction addresses and encodings are set aside: shows that a template or header kernel a new translation unit
instantiates is the code another object already has (tools/sass_counts.py keys by name and cannot tell two such copies
apart).   python tools/sass_same.py build/rt_scene.o build/rt_adaptive.o"""
import re
import subprocess
import sys


def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    cur, code = None, {}
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            code[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if cur and m:
            code[cur].append(m.group(1))
    return code


a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
shared = sorted(set(a) & set(b))
names = subprocess.run(["c++filt"], input="\n".join(shared), capture_output=True, text=True).stdout.splitlines()
for k, d in zip(shared, names):
    print(f"{'same   ' if a[k] == b[k] else 'DIFFERS'} {len(a[k]):6d} {len(b[k]):6d}  {d}")
