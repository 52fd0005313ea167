"""Per-kernel SASS instruction counts (cuobjdump -sass, padding included) and the ptxas register / spill lines of the
Makefile's build/*.ptxas.log, by demangled name, to check that a change leaves existing kernels' code alone without a
profiler:  python tools/sass_counts.py raytracing_renderer_cuda_b200/librt_b200.so [build] > counts.txt"""
import re, subprocess, sys
lib = sys.argv[1]
out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
cur, counts = None, {}
for line in out.splitlines():
    m = re.match(r"\s+Function : (\S+)", line)
    if m:
        cur = m.group(1); counts[cur] = 0; continue
    if cur and re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+\S", line):
        counts[cur] += 1
names = list(counts)
dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
for n, d in sorted(zip(names, dem), key=lambda t: t[1]):
    print(f"{counts[n]:7d} {d}")
if len(sys.argv) > 2:
    import glob

    rows, cur = [], None
    for f in sorted(glob.glob(sys.argv[2] + "/*.ptxas.log")):
        for line in open(f):
            m = re.search(r"Compiling entry function '(\S+)'", line)
            if m:
                cur = m.group(1)
                continue
            m = re.search(r"(Used \d+ registers.*|\d+ bytes stack frame.*)", line)
            if m and cur:
                rows.append((cur, m.group(1).strip()))
    keys = sorted(set(r[0] for r in rows))
    dm = dict(zip(keys, subprocess.run(["c++filt"], input="\n".join(keys), capture_output=True, text=True).stdout.splitlines()))
    for line in sorted(set(f"ptxas {dm[k]} :: {v}" for k, v in rows)):
        print(line)
