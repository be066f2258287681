"""Per-kernel SASS comparison of two builds of libnint.so: which kernel symbols compile to identical instructions, which
differ, which are missing and which are new (demangled).  Needs only cuobjdump, no GPU.

    python tools/sass_compare.py old/libnint.so nasa_niswan_b200/libnint.so
"""
import re
import subprocess
import sys



def funcs(lib):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    d = {}; cur = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m: cur = m.group(1); d[cur] = []; continue
        if cur and re.match(r"\s*/\*[0-9a-f]{4}\*/", line):
            d[cur].append(re.sub(r"\s*/\*[0-9a-f]{4}\*/", "", line).split(";")[0].strip())
    return d


a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
same = [k for k in a if k in b and a[k] == b[k]]
diff = [k for k in a if k in b and a[k] != b[k]]
gone = [k for k in a if k not in b]
new = [k for k in b if k not in a]
print(f"parent {len(a)} kernels; identical {len(same)}; differ {len(diff)}; missing {len(gone)}; new {len(new)}")
for k in diff:
    print("DIFF", k)
for k in gone:
    print("GONE", k)
for k in new:
    print("NEW ", subprocess.run(["c++filt", k], capture_output=True, text=True).stdout.strip())
