"""Per-function SASS comparison of two object files (addresses and comments stripped)."""
import re, subprocess, sys
def funcs(obj):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); res[cur] = []; continue
        if cur and re.match(r"\s*/\*[0-9a-f]{4}\*/", line):
            ins = re.sub(r"/\*[0-9a-f]{4}\*/", "", line).split(";")[0].strip()
            res[cur].append(ins)
    return res
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
pat = sys.argv[3] if len(sys.argv) > 3 else ""
common = sorted(k for k in a if k in b and pat in k)
same = [k for k in common if a[k] == b[k]]
diff = [k for k in common if a[k] != b[k]]
print(f"parent functions {len(a)}, branch functions {len(b)}, compared (matching '{pat}') {len(common)}, identical {len(same)}, different {len(diff)}")
print("only in parent:", sorted(set(a) - set(b)))
print("only in branch:", sorted(k for k in set(b) - set(a)))
for k in diff: print("DIFF", k)
